"""Sort by several key columns on the GPU: lsb_lexsort_device, DistributedSorter.lexsort_device and lsb.lexsort -- needs
a B200.

Every result is compared bit for bit with np.lexsort over each column's dense ranks, taken from numpy's own comparison of
the typed values (tests/lexsort_ref.py), which shares no code with order_key / order_key_narrow.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import lexsort_ref as R  # noqa: E402
import patterns as P  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from test_gpu_patterns import _expected_skips  # noqa: E402
from test_lexsort_cpu import order  # noqa: E402

TL, OP, NS, DESC = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP, L.FLAG_DESCENDING
I64, F64 = L.FLAG_KEY_I64, L.FLAG_KEY_F64
ERR_ARG = -1


def _planned_passes(names, radix):
    return sum(r[3] for r in H.lexsort_rounds([R.WIDTH[x] for x in names], radix))


def _check(cols, names, desc, flags=0, radix=16, vals=None, sorter=None):
    """lexsort_device of the bit-pattern columns `cols` (types `names`, least significant first); returns (out, stats)"""
    n = len(cols[0])
    ts = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    before = [t.clone() for t in ts]
    s = sorter or lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags)
    try:
        out, st = s.lexsort_device(ts, vals, descending=list(desc))
        want = R.reference(cols, names, desc)
        what = (names, desc, flags, s.radix_bits, n)
        got = out.view(torch.int64).cpu().numpy()
        if vals is None:
            assert out.dtype == torch.int64 and np.array_equal(got, want), what
        else:
            assert out.dtype == vals.dtype and np.array_equal(got, vals.view(torch.int64).cpu().numpy()[want]), what
        assert st.passes == _planned_passes(names, s.radix_bits), what
        for t, b in zip(ts, before):  # the columns are never rewritten
            assert n == 0 or torch.equal(t.view(torch.uint8), b.view(torch.uint8)), what
        return out, st
    finally:
        if sorter is None:
            s.close()


# ---- 1. types and directions ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", R.NAMES)
def test_types_and_directions(name):
    """every type as the primary and as the secondary key, each column in both directions, special values throughout"""
    n = (1 << 17) + 3
    for other in ("int16", "float64", "float32", "bfloat16"):
        for names in ((other, name), (name, other)):
            cols = [R.special_mix(n, names[0], seed=1), R.special_mix(n, names[1], seed=2)]  # half specials: many ties
            for desc in ((False, False), (True, False), (False, True), (True, True)):
                _check(cols, names, desc)


# ---- 2. rounds, ties, pass shapes, radices ------------------------------------------------------------------------------
ROUND_MIXES = [
    ("int32", "float32"),                                   # 64 bits: one round
    ("bfloat16", "int16", "int32"),                         # 64 bits: one round
    ("int32", "float32", "uint16"),                         # 80 bits: 64 + 16
    ("int16", "int16", "int16", "int16", "float16"),       # 4 x 16 + 16: the column limit
    ("uint16", "float64", "int32", "int32"),                # 16 | 64 | 64
    ("int64", "int64"),
    ("float64", "int64", "uint64"),
    ("float16", "uint32", "bfloat16", "int64", "float32", "int16"),  # 64 | 64 | 48
]


@pytest.mark.parametrize("mix", range(len(ROUND_MIXES)))
def test_rounds_and_ties(mix):
    """1-6 columns with round boundaries on both sides of 64 bits; few distinct values per column, so the lower
    columns decide most ties, with random directions"""
    names = ROUND_MIXES[mix]
    n = (1 << 19) + 11
    rng = np.random.default_rng(mix)
    cols = [R.few_values(n, x, k=int(rng.integers(2, 9)), seed=10 * mix + c) for c, x in enumerate(names)]
    for trial in range(3):
        _check(cols, names, [bool(d) for d in rng.integers(0, 2, len(names))])


@pytest.mark.parametrize("radix", [8, 11, 13, 16])
@pytest.mark.parametrize("flags", [0, OP, TL, NS])
def test_pass_shapes_and_radices(flags, radix):
    n = P.SUPERTILE + 1
    for mix in (0, 2, 5, 7):
        names = ROUND_MIXES[mix]
        cols = [R.few_values(n, x, k=5, seed=c) if c < len(names) - 1 else R.special_mix(n, x, seed=c)
                for c, x in enumerate(names)]
        _check(cols, names, [c % 2 == 1 for c in range(len(names))], flags, radix)


@pytest.mark.parametrize("n", [0, 1, 31, 33, (1 << 20) - 5, (1 << 24) + 13])
def test_sizes(n):
    names = ("int64", "float32", "bfloat16")
    cols = [R.special_mix(n, names[0], seed=1), R.few_values(n, names[1], 20, seed=2), R.few_values(n, names[2], 7, seed=3)]
    for flags in ((0, OP, TL) if n < (1 << 24) else (0,)):
        _check(cols, names, (False, True, False), flags)


# ---- 3. stats -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, OP, TL, NS])
def test_skipped_on_low_cardinality(flags):
    """int64 columns of 256 values: in every round the digits above the low byte are constant and skipped"""
    n = P.SUPERTILE + 1
    rng = np.random.default_rng(3)
    names = ("int64", "int64", "int32", "int32")
    cols = [rng.integers(0, 256, n).astype(np.uint64) for _ in range(2)] + \
           [rng.integers(-3, 3, n).astype(np.int32).view(np.uint32) for _ in range(2)]
    _, st = _check(cols, names, (False, True, False, False), flags)
    words = [order(cols[0], "int64", False), order(cols[1], "int64", True),
             order(cols[2], "int32", False) | order(cols[3], "int32", False) << np.uint64(32)]
    assert st.skipped == sum(_expected_skips(w, flags) for w in words)
    assert (st.skipped > 0) == (not flags & NS) and st.passes == 12


# ---- 4. outputs ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("vals", ["int64", "float64"])
def test_vals_gathered(vals):
    n = P.SUPERTILE + 1
    rng = np.random.default_rng(5)
    if vals == "int64":
        v = torch.from_numpy(rng.integers(-(1 << 63), (1 << 63) - 1, n, dtype=np.int64)).cuda()
    else:  # NaN payloads of both signs survive the gather
        v = torch.from_numpy(R.special_mix(n, "float64", seed=6).view(np.float64)).cuda()
    names = ("uint16", "float64", "int32")
    cols = [R.few_values(n, x, 9, seed=c) for c, x in enumerate(names)]
    for flags in (0, OP, TL):
        with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
            out, _ = _check(cols, names, (True, False, True), sorter=s, vals=v)
            given = torch.empty_like(v)
            out2, _ = s.lexsort_device([R.to_device(torch, b, x) for b, x in zip(cols, names)], v, vals_out=given,
                                       descending=[True, False, True])
            assert out2 is given and torch.equal(out.view(torch.int64), given.view(torch.int64))


@pytest.mark.parametrize("name", R.NAMES)
def test_one_column_is_the_sort(name):
    """a one-column lexsort returns exactly the indices of sort_device / sort_device_typed on that column"""
    n = P.SUPERTILE + 1
    bits = R.special_mix(n, name, seed=8)
    t = R.to_device(torch, bits, name)
    for descending in (False, True):
        for flags in (0, OP, TL):
            wide = {"uint64": 0, "int64": I64, "float64": F64}
            base = flags | (DESC if descending else 0)
            kw = {"flags": base | wide[name]} if name in wide else {"flags": base, "key_dtype": getattr(torch, name)}
            with lsb.DistributedSorter(n, ranks=1, **kw) as s:
                _, want, st1 = s.sort_device(t, keys_out=False)
            with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
                got, st2 = s.lexsort_device([t], descending=descending)
            assert torch.equal(got, want) and st1.passes == st2.passes, (name, descending, flags)


# ---- 5. the C entry point ------------------------------------------------------------------------------------------------
def test_c_level_refusals():
    n = 10007
    f32 = R.to_device(torch, R.special_mix(n, "float32", seed=12), "float32")
    i64 = R.to_device(torch, R.special_mix(n, "int64", seed=13), "int64")
    vin = torch.arange(n, dtype=torch.int64, device="cuda")
    out = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    host = np.zeros(n, dtype=np.int64)
    big = torch.empty(4 * n, dtype=torch.int64, device="cuda")  # a 4-byte column at its start, vals_out inside it
    F32 = L.NARROW_KEY_TYPES["float32"]

    def cols(*spec):
        a = (L.KeyColumn * max(len(spec), 1))()
        for c, (p, kt, fl) in enumerate(spec):
            a[c].keys, a[c].key_type, a[c].flags = p, kt, fl
        return a

    good = [(i64.data_ptr(), 0, I64), (f32.data_ptr(), F32, DESC)]
    with lsb.DistributedSorter(n, ranks=1) as s:
        Lb, ctx = s._L, s._ctx

        def call(spec, k=None, vi=None, vo=out.data_ptr(), count=n):
            return Lb.lsb_lexsort_device(ctx, cols(*spec), len(spec) if k is None else k, vi, vo, count, None, None)

        cases = {  # what -> (call, a word the message must hold)
            "no columns": (lambda: call(good, k=0), "num_columns"),
            "negative num_columns": (lambda: call(good, k=-1), "num_columns"),
            "columns NULL": (lambda: Lb.lsb_lexsort_device(ctx, None, 1, None, out.data_ptr(), n, None, None), "columns"),
            "unknown key_type 8": (lambda: call([good[0], (f32.data_ptr(), 8, 0)]), "column 1"),
            "unknown key_type 2^31": (lambda: call([(f32.data_ptr(), 1 << 31, 0)]), "column 0"),
            "KEY_I64 on a narrow column": (lambda: call([good[0], (f32.data_ptr(), F32, I64)]), "column 1"),
            "KEY_I64 | KEY_F64": (lambda: call([(i64.data_ptr(), 0, I64 | F64)]), "column 0"),
            "another flag bit": (lambda: call([good[0], (i64.data_ptr(), 0, 128)]), "column 1"),
            "ONE_PASS as a column flag": (lambda: call([(f32.data_ptr(), F32, OP)]), "column 0"),
            "count != here": (lambda: call(good, count=n - 1), "count"),
            "keys NULL": (lambda: call([good[0], (None, F32, 0)]), "column 1"),
            "misaligned 4-byte column": (lambda: call([good[0], (f32.data_ptr() + 2, F32, 0)]), "column 1"),
            "misaligned 8-byte column": (lambda: call([(i64.data_ptr() + 4, 0, 0)]), "column 0"),
            "host memory column": (lambda: call([good[0], (host.ctypes.data, 0, 0)]), "column 1"),
            "the context's own shard": (lambda: call([good[0], (s.device_ptr(), 0, 0)]), "column 1"),
            "misaligned vals_in": (lambda: call(good, vi=vin.data_ptr() + 4), "vals_in"),
            "vals_out NULL": (lambda: call(good, vo=None), "vals_out"),
            "misaligned vals_out": (lambda: call(good, vo=out.data_ptr() + 4), "vals_out"),
            "vals_out overlaps vals_in": (lambda: call(good, vi=out.data_ptr() + 8 * (n - 1)), "vals_in"),
            "vals_out overlaps a column": (lambda: call(good, vo=i64.data_ptr() + 8 * (n - 1)), "column 0"),
            "vals_out overlaps a 4-byte column": (lambda: call([good[0], (big.data_ptr(), F32, 0)], vo=big.data_ptr() + 8 * ((4 * n - 1) // 8)),
                                                  "column 1"),
        }
        for what, (fn, word) in cases.items():
            assert fn() == ERR_ARG, what
            assert word in Lb.lsb_last_error(ctx).decode(), (what, Lb.lsb_last_error(ctx).decode())
        assert call(good) == 0
        want = R.reference([R.special_mix(n, "int64", seed=13), R.special_mix(n, "float32", seed=12)],
                           ["int64", "float32"], [False, True])
        assert np.array_equal(out[:n].cpu().numpy(), want)
        # vals_out from the next 8-byte boundary after a 4-byte column: the real widths do not overlap
        assert call([good[0], (big.data_ptr(), F32, DESC)], vo=big.data_ptr() + 8 * ((4 * n + 7) // 8)) == 0
    for flags in (I64, F64, DESC, I64 | DESC):  # the order comes from the columns only
        with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
            spec = cols(*good)
            assert s._L.lsb_lexsort_device(s._ctx, spec, 2, None, out.data_ptr(), n, None, None) == ERR_ARG
            assert b"key-order" in s._L.lsb_last_error(s._ctx)
    with lsb.DistributedSorter(2 * n, world_size=2, world_rank=0) as s:  # one GPU only, refused before the comm state
        spec = cols(*good)
        assert s._L.lsb_lexsort_device(s._ctx, spec, 2, None, out.data_ptr(), n, None, None) == ERR_ARG
        assert b"one GPU" in s._L.lsb_last_error(s._ctx)
    with lsb.DistributedSorter(0, ranks=1) as s:  # count 0: no device pointer is looked at
        st = L.Stats()
        spec = cols((None, 0, F64), (12345, F32, DESC))
        assert s._L.lsb_lexsort_device(s._ctx, spec, 2, 8, None, 0, None, ctypes.byref(st)) == 0
        assert st.passes == 4 + 2 and st.elements == 0


def test_waits_for_the_callers_stream():
    n = (1 << 20) + 7
    names = ("int32", "float64")
    cols = [R.few_values(n, "int32", 30, seed=1), R.special_mix(n, "float64", seed=2)]
    new = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    keys = [torch.zeros_like(t) for t in new]
    side = torch.cuda.Stream()
    with lsb.DistributedSorter(n, ranks=1) as s:
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(100_000_000)  # tens of ms on the side stream before the columns are written
            for k, t in zip(keys, new):
                k.copy_(t)
        out, _ = s.lexsort_device(keys, stream=side)  # no synchronise in between
    assert np.array_equal(out.cpu().numpy(), R.reference(cols, names, (False, False)))


# ---- 6. a reused sorter: no call rewrites the context ---------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, OP, TL])
def test_interleaved_with_other_calls(flags):
    n, radix = P.SUPERTILE + 1, 13
    rng = np.random.default_rng(18)
    names = ("float32", "int64", "bfloat16")
    cols = [R.special_mix(n, "float32", 1), R.few_values(n, "int64", 40, seed=2), R.few_values(n, "bfloat16", 5, seed=3)]
    ts = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    keys = torch.from_numpy(rng.integers(0, 1 << 62, n, dtype=np.int64)).cuda().view(torch.uint64)
    offsets = torch.from_numpy(np.concatenate([[0], np.sort(rng.integers(0, n, 99)), [n]]).astype(np.int64)).cuda()

    def lex(s):
        v, st = s.lexsort_device(ts, descending=[False, True, True])
        return v.cpu().numpy(), st.passes, st.skipped

    def device(s):
        k, v, st = s.sort_device(keys)
        return k.view(torch.int64).cpu().numpy(), v.cpu().numpy(), st.passes

    def segments(s):
        k, v, st = s.sort_segments(keys, offsets)
        return k.view(torch.int64).cpu().numpy(), v.cpu().numpy(), st.passes

    def plan(s):
        return s.num_passes(), [s.digit_bits(d) for d in range(s.num_passes())]

    def sorter():
        return lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags)

    with sorter() as s:
        for call in [lex, device, lex, segments, plan, lex, lex, segments, device, plan]:
            got = call(s)
            with sorter() as fresh:
                want = call(fresh)
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), call.__name__
        assert plan(s) == (5, [13, 13, 13, 13, 12])
        v, passes, _ = lex(s)
        assert np.array_equal(v, R.reference(cols, names, (False, True, True))) and passes == _planned_passes(names, radix)


# ---- 7. lsb.lexsort: np.lexsort for CUDA tensors --------------------------------------------------------------------------
def test_oneshot_lexsort():
    n = 100003
    rng = np.random.default_rng(21)
    names = ("uint32", "float16", "int64", "float32")
    cols = [R.few_values(n, x, 6, seed=c) for c, x in enumerate(names)]
    ts = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    for desc in (False, True, [True, False, False, True]):
        d = [desc] * 4 if isinstance(desc, bool) else desc
        want = R.reference(cols, names, d)
        got = lsb.lexsort(ts, descending=desc)
        assert got.dtype == torch.int64 and np.array_equal(got.cpu().numpy(), want), desc
        assert np.array_equal(lsb.lexsort(tuple(ts), descending=desc).cpu().numpy(), want)
    # with no NaNs and one dtype, np.lexsort itself agrees
    x = rng.integers(-5, 5, (3, n)).astype(np.float32)
    t = torch.from_numpy(x).cuda()
    assert np.array_equal(lsb.lexsort(t).cpu().numpy(), np.lexsort(x))
    assert np.array_equal(lsb.lexsort(t.t().contiguous().t()).cpu().numpy(), np.lexsort(x))  # rows not contiguous
    assert np.array_equal(lsb.lexsort(list(t[:, ::2])).cpu().numpy(), np.lexsort(x[:, ::2]))   # strided keys
    vals = torch.from_numpy(rng.standard_normal(n)).cuda()
    assert torch.equal(lsb.lexsort(t, vals=vals), vals[torch.from_numpy(np.lexsort(x)).cuda()])
    assert lsb.lexsort([torch.zeros(0, dtype=torch.int16, device="cuda")]).numel() == 0
    with pytest.raises(ValueError):
        lsb.lexsort([ts[0], ts[1][1:]])
    with pytest.raises(ValueError):
        lsb.lexsort([], descending=True)
