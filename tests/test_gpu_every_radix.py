"""Every radix from 1 to 16, in every pass shape, on inputs where every step decides the output -- needs a B200.

The inputs hold copies of the block tests/test_decisive_cpu.py proves: there every fault of every step of the plan
(skipped, digit read one bit off, bins merged, ties reversed, last digit not clamped, raw bits instead of the order key)
changes the output, so a whole-sort comparison here sees a faulty step even where later steps would hide it on other
data.  Results are compared bit for bit with references that share no code with order_key: numpy's stable argsort of
the typed keys (key_orders / narrow_keys), np.lexsort over dense ranks (lexsort_ref), and pass by pass with the C
oracle on order_key(keys).
"""
import collections
import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import decisive as D  # noqa: E402
import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import lexsort_ref as R  # noqa: E402
import narrow_keys as NK  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from oracle import oracle as O  # noqa: E402
from test_gpu_patterns import _assert_same, _expected_skips  # noqa: E402

TL, OP, NS, DESC = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP, L.FLAG_DESCENDING
RADICES = list(range(1, 17))
SHAPES = [0, NS, OP, TL, TL | OP]
PASS_SHAPES = [0, OP, TL, TL | OP]
SHAPE_IDS = {0: "default", NS: "no_skip", OP: "one_pass", TL: "two_level", TL | OP: "two_level+one_pass"}


# ---- sorters: one per (count, radix, flags), reused across calls; a few dozen alive at most ----------------------------------
_SORTERS = collections.OrderedDict()


def _sorter(n, radix, flags):
    key = (n, radix, flags)
    if key in _SORTERS:
        _SORTERS.move_to_end(key)
        return _SORTERS[key]
    while len(_SORTERS) >= 24:
        _SORTERS.popitem(last=False)[1].close()
    _SORTERS[key] = lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags)
    return _SORTERS[key]


@pytest.fixture(scope="module", autouse=True)
def _close_sorters():
    yield
    while _SORTERS:
        _SORTERS.popitem()[1].close()


# ---- data and references, cached per (plan, count) ------------------------------------------------------------------------
@functools.lru_cache(maxsize=8)
def _records(order, n):
    plan = D.sort_plan(*D.WIDE_ORDERS[order], n=n)
    a = np.zeros(n, dtype=L.ELT)
    a["key"] = plan.given["raw"]
    a["val"] = np.arange(n, dtype=np.uint64)
    return a, KO.reference(a, KO.ORDERS[order])


@functools.lru_cache(maxsize=16)
def _narrow(name, descending, n):
    raw = D.sort_plan(name, descending, n=n).given["raw"]
    return raw, NK.argsort(raw, name, descending)


@functools.lru_cache(maxsize=8)
def _lexsort(mix, n):
    names, desc = D.LEXSORTS[mix]
    cols = D.lexsort_plan(names, desc, n=n).given["cols"]
    return cols, R.reference(cols, names, desc)


@functools.lru_cache(maxsize=4)
def _segments(name, descending, segbits, n):
    g = D.segment_plan(name, descending, segbits, n=n).given
    perm = np.lexsort((R.ranks(g["raw"], name, descending), g["seg"]))
    return g["raw"], g["offsets"], perm, perm - g["offsets"][g["seg"][perm]]


def _params(shapes=SHAPES):
    return [pytest.param(r, f, id=f"r{r}-{SHAPE_IDS[f]}") for r in RADICES for f in shapes]


# ---- 1. upload + my_sort, and the step counts ------------------------------------------------------------------------------
@pytest.mark.parametrize("radix,shape", _params())
def test_records(radix, shape):
    n = D.gpu_count(radix)
    for order in D.WIDE_ORDERS:
        korder = KO.ORDERS[order]
        a, want = _records(order, n)
        s = _sorter(n, radix, korder | shape)
        s.upload(a)
        st = s.my_sort()
        _assert_same(s.download(), want, order, radix, shape)
        assert st.passes == -(-64 // radix), (order, radix, shape)
        assert st.skipped == _expected_skips(KO.order_key(a["key"], korder), shape, radix), (order, radix, shape)


# ---- 2. pass by pass against the oracle on order_key(keys) ----------------------------------------------------------------
@pytest.mark.parametrize("radix,shape", _params(PASS_SHAPES))
def test_each_pass(radix, shape):
    n = D.gpu_count(radix)
    for order in ("u64", "f64_desc"):
        korder = KO.ORDERS[order]
        a, _ = _records(order, n)
        cur = a.copy()
        cur["key"] = KO.order_key(a["key"], korder)  # the oracle sorts order_key as plain uint64
        s = _sorter(n, radix, korder | shape)
        s.upload(a)
        assert s.num_passes() == -(-64 // radix)
        for p in range(s.num_passes()):
            want, counts, starts, _ = O.one_pass(cur, n, 1, radix, p)
            nb = 1 << s.digit_bits(p)  # the last digit is clamped to the 64 bits of the key
            what = (order, radix, shape, p)
            assert nb == 1 << H.plan_pass(radix, p)[1] and counts[0, nb:].sum() == 0, what
            assert (s.histogram(p) == counts[0, :nb]).all(), what
            assert (s.starts(p) == starts[:nb, 0]).all(), what
            s.global_shuffle(p)
            got = s.download()
            assert np.array_equal(got["val"], want["val"]), what
            assert np.array_equal(got["key"], a["key"][got["val"].astype(np.int64)]), what
            cur = want


# ---- 3. narrow keys through lsb_sort_device_typed ----------------------------------------------------------------------------
@pytest.mark.parametrize("radix,shape", _params())
def test_narrow_keys(radix, shape):
    n = D.gpu_count(radix)
    out = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    for name in NK.NAMES:
        desc = D.narrow_descending(name, radix)
        raw, perm = _narrow(name, desc, n)
        keys = NK.to_device(torch, raw, name)
        s = _sorter(n, radix, shape | (DESC if desc else 0))
        st = L.Stats()
        kout, vout = out[:n].view(keys.dtype)[:n], out[n:]
        assert s._L.lsb_sort_device_typed(s._ctx, NK.KEY_TYPE[name], keys.data_ptr(), None, kout.data_ptr(),
                                          vout.data_ptr(), n, None, ctypes.byref(st)) == 0, s._L.lsb_last_error(s._ctx)
        what = (name, desc, radix, shape)
        assert np.array_equal(NK.bits_of(torch, kout), raw[perm]), what
        assert np.array_equal(vout.cpu().numpy(), perm), what
        assert st.passes == -(-NK.BITS[name] // radix), what


# ---- 4. lexsort rounds of 16, 32, 48 and 64 bits, and 64 | 64 | 48 ---------------------------------------------------------------
@pytest.mark.parametrize("radix,shape", _params())
def test_lexsort(radix, shape):
    n = D.gpu_count(radix)
    s = _sorter(n, radix, shape)
    for mix, (names, desc) in enumerate(D.LEXSORTS):
        cols, want = _lexsort(mix, n)
        out, st = s.lexsort_device([R.to_device(torch, b, x) for b, x in zip(cols, names)], descending=list(desc))
        what = (names, radix, shape)
        assert np.array_equal(out.cpu().numpy(), want), what
        assert st.passes == sum(r[3] for r in H.lexsort_rounds([R.WIDTH[x] for x in names], radix)), what


# ---- 5. segments: 2^(radix + 1) of them, two segment passes at every radix ----------------------------------------------------
@pytest.mark.parametrize("radix,shape", _params())
def test_segments(radix, shape):
    n = D.gpu_count(radix)
    segbits = D.segment_bits(radix)
    for name, desc in D.SEGMENT_KEYS:
        raw, off, perm, local = _segments(name, desc, segbits, n)
        offsets = torch.from_numpy(off).cuda()
        what = (name, desc, radix, shape)
        passes = -(-R.WIDTH[name] // radix) + H.segsort_layout(n, len(off) - 1, radix)[3]
        assert H.segsort_layout(n, len(off) - 1, radix)[3] == 2
        if R.WIDTH[name] == 64:
            s = _sorter(n, radix, shape | KO.F64 | (DESC if desc else 0))
            keys = torch.from_numpy(raw.view(np.int64)).cuda().view(torch.float64)
            k, v, st = s.sort_segments(keys, offsets)
            assert np.array_equal(k.view(torch.int64).cpu().numpy().view(np.uint64), raw[perm]), what
            assert np.array_equal(v.cpu().numpy(), perm) and st.passes == passes, what
            _, v, _ = s.sort_segments(keys, offsets, keys_out=False, local_index=True)
            assert np.array_equal(v.cpu().numpy(), local), what
            continue
        s = _sorter(n, radix, shape | (DESC if desc else 0))
        keys = NK.to_device(torch, raw, name)
        out = torch.empty(2 * n, dtype=torch.int64, device="cuda")
        kout, vout = out[:n].view(keys.dtype)[:n], out[n:]
        for flags, want in ((0, perm), (L.SEG_LOCAL_INDEX, local)):
            st = L.Stats()
            assert s._L.lsb_sort_segments_device_typed(s._ctx, NK.KEY_TYPE[name], keys.data_ptr(), None, kout.data_ptr(),
                                                       vout.data_ptr(), n, offsets.data_ptr(), len(off) - 1, flags, None,
                                                       ctypes.byref(st)) == 0, s._L.lsb_last_error(s._ctx)
            assert np.array_equal(NK.bits_of(torch, kout), raw[perm]), what
            assert np.array_equal(vout.cpu().numpy(), want) and st.passes == passes, what
