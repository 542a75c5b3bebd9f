"""Distinct keys and rows on the GPU: lsb_unique_device, DistributedSorter.unique_device, lsb.unique and
lsb.unique_consecutive -- needs a B200.

Every result is compared bit for bit with tests/unique_ref.py (groups from numpy's own comparison of the typed values)
or with torch, and every call checks that the columns were not rewritten.
"""
import ctypes
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import lexsort_ref as R  # noqa: E402
import patterns as P  # noqa: E402
import unique_ref as U  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from test_gpu_lexsort import ROUND_MIXES  # noqa: E402

TL, OP, NS, DESC = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP, L.FLAG_DESCENDING
I64, F64 = L.FLAG_KEY_I64, L.FLAG_KEY_F64
ERR_ARG = -1
TILE = 2048         # positions per tile of unique_tile_kernel (lsb_unique.cuh)
SENTINEL = -7


def _check(cols, names, desc=None, consecutive=False, flags=0, radix=16, sorter=None, outputs=(True, True, True)):
    """unique_device of the bit-pattern columns `cols` (types `names`, least significant first) against the reference;
    every output not asked for is False, and index / counts start as a sentinel that must survive past entry U"""
    n = len(cols[0])
    desc = list(desc) if desc is not None else [False] * len(cols)
    ts = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    before = [t.clone() for t in ts]
    outs = [torch.full((n,), SENTINEL, dtype=torch.int64, device="cuda") if want else False for want in outputs]
    s = sorter or lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags)
    try:
        index, inverse, counts, u, st = s.unique_device(ts, descending=desc, consecutive=consecutive, index_out=outs[0],
                                                        inverse_out=outs[1], counts_out=outs[2])
        want = U.reference(cols, names, desc, consecutive)
        what = (names, desc, consecutive, flags, s.radix_bits, n)
        assert u == len(want[0]), what
        for got, w, full in ((index, want[0], True), (inverse, want[1], False), (counts, want[2], True)):
            if got is None:
                continue
            g = got.cpu().numpy()
            assert np.array_equal(g[:len(w)], w), what
            assert not full or (g[len(w):] == SENTINEL).all(), what
        rounds = H.lexsort_rounds([R.WIDTH[x] for x in names], s.radix_bits)
        assert st.passes == (0 if consecutive else sum(r[3] for r in rounds)), what
        for t, b in zip(ts, before):
            assert n == 0 or torch.equal(t.view(torch.uint8), b.view(torch.uint8)), what
        return u, st
    finally:
        if sorter is None:
            s.close()


# ---- 1. types, directions, modes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", R.NAMES)
def test_types_directions_and_modes(name):
    n = (1 << 16) + 3
    for bits in (R.special_mix(n, name, seed=1), R.few_values(n, name, 9, seed=2)):
        for desc, consecutive in itertools.product((False, True), (False, True)):
            _check([bits], [name], [desc], consecutive)
    runs = np.repeat(R.few_values(4000, name, 5, seed=3), np.random.default_rng(4).integers(1, 40, 4000))  # real runs
    for consecutive in (False, True):
        _check([runs], [name], None, consecutive)


# ---- 2. rounds, pass shapes, radices --------------------------------------------------------------------------------------
@pytest.mark.parametrize("mix", range(len(ROUND_MIXES)))
def test_round_mixes(mix):
    """1 to 3 rounds, so 0 to 2 gather-flag launches; few values per column, so every column decides some heads"""
    names = ROUND_MIXES[mix]
    n = (1 << 18) + 11
    rng = np.random.default_rng(mix)
    cols = [R.few_values(n, x, k=int(rng.integers(2, 5)), seed=10 * mix + c) for c, x in enumerate(names)]
    for consecutive in (False, True):
        _check(cols, names, [bool(d) for d in rng.integers(0, 2, len(names))], consecutive)
    # consecutive runs in every column at once
    order = np.lexsort([R.ranks(c, x) for c, x in zip(cols, names)])
    _check([c[order] for c in cols], names, None, True)


@pytest.mark.parametrize("radix", [8, 11, 13, 16])
@pytest.mark.parametrize("flags", [0, OP, TL, NS])
def test_pass_shapes_and_radices(flags, radix):
    n = P.SUPERTILE + 1
    for mix in (0, 2, 7):
        names = ROUND_MIXES[mix]
        cols = [R.few_values(n, x, k=4, seed=c) for c, x in enumerate(names)]
        _check(cols, names, [c % 2 == 1 for c in range(len(names))], False, flags, radix)
    _check([R.special_mix(n, "float64", seed=5)], ["float64"], None, False, flags, radix)


# ---- 3. layouts -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 2, 31, 33, TILE - 1, TILE, TILE + 1, 3 * TILE + 17, (1 << 20) + 5])
def test_sizes(n):
    for name in ("int64", "float32", "uint16"):
        bits = R.few_values(n, name, 3, seed=n % 97)
        for consecutive in (False, True):
            _check([bits], [name], None, consecutive)
            _check([bits, R.few_values(n, "float64", 2, seed=1)], [name, "float64"], None, consecutive)


def test_layouts():
    n = 5 * TILE + 77
    rng = np.random.default_rng(9)
    distinct = rng.permutation(n).astype(np.uint64)
    cases = {
        "all equal": np.full(n, 42, dtype=np.uint64),
        "all distinct": distinct,
        "all distinct, sorted": np.sort(distinct),
        # runs crossing tile boundaries: run lengths around the tile size
        "long runs": np.repeat(np.arange(8, dtype=np.uint64), [TILE - 1, TILE + 1, 1, 2 * TILE, 3, TILE, 50, 0])[:n],
        # the first occurrence of a group is the last input element
        "last is new": np.concatenate([np.full(n - 1, 5, dtype=np.uint64), [3]]).astype(np.uint64),
    }
    for what, bits in cases.items():
        for consecutive in (False, True):
            u, _ = _check([bits], ["uint64"], None, consecutive)
            if what == "all equal":
                assert u == 1
            if what.startswith("all distinct"):
                assert u == len(bits)


def test_every_subset_of_outputs():
    n = 3 * TILE + 5
    cols = [R.few_values(n, "int32", 50, seed=1), R.few_values(n, "float64", 3, seed=2), R.special_mix(n, "bfloat16", 3)]
    names = ["int32", "float64", "bfloat16"]
    for outputs in itertools.product((False, True), repeat=3):
        for consecutive in (False, True):
            _check(cols, names, [True, False, True], consecutive, outputs=outputs)


# ---- 4. a kept sorter, streams ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, OP, TL])
def test_kept_sorter_interleaved(flags):
    n, radix = P.SUPERTILE + 1, 13
    rng = np.random.default_rng(18)
    keys = torch.from_numpy(rng.integers(0, 1 << 62, n, dtype=np.int64)).cuda().view(torch.uint64)
    lexcols = [R.to_device(torch, R.few_values(n, "int64", 40, seed=2), "int64")]
    calls = [(["int64"], False), (["float32", "int16"], True), ("sort", None), (["float64", "int32", "uint16"], False),
             ("lexsort", None), (["bfloat16"], True), (["uint64", "uint64"], False), ("sort", None), (["int16"], False)]
    with lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags) as s:
        for c, (what, consecutive) in enumerate(calls):
            if what == "sort":
                k, v, _ = s.sort_device(keys)
                k = k.view(torch.int64)  # keys below 2^62: the same order
                assert torch.equal(k, keys.view(torch.int64)[v]) and bool((k[1:] >= k[:-1]).all())
            elif what == "lexsort":
                v, _ = s.lexsort_device(lexcols)
                assert np.array_equal(v.cpu().numpy(), R.reference([R.few_values(n, "int64", 40, seed=2)], ["int64"], [False]))
            else:
                cols = [R.few_values(n, x, 6, seed=c + j) for j, x in enumerate(what)]
                _check(cols, what, None, consecutive, sorter=s)


def test_waits_for_the_callers_stream():
    n = (1 << 20) + 7
    bits = R.few_values(n, "float32", 30, seed=1)
    new = R.to_device(torch, bits, "float32")
    key = torch.zeros_like(new)
    side = torch.cuda.Stream()
    with lsb.DistributedSorter(n, ranks=1) as s:
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(100_000_000)  # tens of ms on the side stream before the column is written
            key.copy_(new)
        index, inverse, counts, u, _ = s.unique_device([key], stream=side)  # no synchronise in between
    want = U.reference([bits], ["float32"])
    assert u == len(want[0]) and np.array_equal(index[:u].cpu().numpy(), want[0])
    assert np.array_equal(inverse.cpu().numpy(), want[1]) and np.array_equal(counts[:u].cpu().numpy(), want[2])


# ---- 5. the C entry point ------------------------------------------------------------------------------------------------
def test_c_level_refusals():
    n = 10007
    f32 = R.to_device(torch, R.special_mix(n, "float32", seed=12), "float32")
    i64 = R.to_device(torch, R.special_mix(n, "int64", seed=13), "int64")
    outs = [torch.empty(n, dtype=torch.int64, device="cuda") for _ in range(3)]
    wide = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    big = torch.empty(4 * n, dtype=torch.int64, device="cuda")  # a 4-byte column at its start, counts_out inside it
    host = np.zeros(n, dtype=np.int64)
    F32 = L.NARROW_KEY_TYPES["float32"]

    def cols(*spec):
        a = (L.KeyColumn * max(len(spec), 1))()
        for c, (p, kt, fl) in enumerate(spec):
            a[c].keys, a[c].key_type, a[c].flags = p, kt, fl
        return a

    good = [(i64.data_ptr(), 0, I64), (f32.data_ptr(), F32, DESC)]
    ptrs = [t.data_ptr() for t in outs]
    u = ctypes.c_int64(-1)
    with lsb.DistributedSorter(n, ranks=1) as s:
        Lb, ctx = s._L, s._ctx

        def call(spec, k=None, uf=0, o=None, count=n, num=ctypes.byref(u)):
            o = ptrs if o is None else o
            return Lb.lsb_unique_device(ctx, cols(*spec), len(spec) if k is None else k, uf, *o, count, num, None, None)

        cases = {  # what -> (call, a word the message must hold)
            "no columns": (lambda: call(good, k=0), "num_columns"),
            "columns NULL": (lambda: Lb.lsb_unique_device(ctx, None, 1, 0, *ptrs, n, ctypes.byref(u), None, None), "columns"),
            "unknown key_type": (lambda: call([good[0], (f32.data_ptr(), 8, 0)]), "column 1"),
            "KEY_I64 on a narrow column": (lambda: call([good[0], (f32.data_ptr(), F32, I64)]), "column 1"),
            "KEY_I64 | KEY_F64": (lambda: call([(i64.data_ptr(), 0, I64 | F64)]), "column 0"),
            "unknown unique_flags 2": (lambda: call(good, uf=2), "unique_flags"),
            "unknown unique_flags 2^31": (lambda: call(good, uf=1 << 31), "unique_flags"),
            "count != here": (lambda: call(good, count=n - 1), "count"),
            "num_unique NULL": (lambda: call(good, num=None), "num_unique"),
            "keys NULL": (lambda: call([good[0], (None, F32, 0)]), "column 1"),
            "misaligned column": (lambda: call([good[0], (f32.data_ptr() + 2, F32, 0)]), "column 1"),
            "host memory column": (lambda: call([(host.ctypes.data, 0, 0)]), "column 0"),
            "the context's own shard as a column": (lambda: call([(s.device_ptr(), 0, 0)]), "column 0"),
            "misaligned index_out": (lambda: call(good, o=[ptrs[0] + 4, ptrs[1], ptrs[2]]), "index_out"),
            "host inverse_out": (lambda: call(good, o=[ptrs[0], host.ctypes.data, ptrs[2]]), "inverse_out"),
            "counts_out in the shard": (lambda: call(good, o=[None, None, s.device_ptr()]), "counts_out"),
            "inverse_out overlaps index_out": (lambda: call(good, o=[wide.data_ptr(), wide.data_ptr() + 8 * (n - 1), None]),
                                               "index_out"),
            "counts_out overlaps inverse_out": (lambda: call(good, o=[None, wide.data_ptr(), wide.data_ptr() + 8]),
                                                "inverse_out"),
            "index_out overlaps a column": (lambda: call(good, o=[i64.data_ptr() + 8 * (n - 1), None, None]), "column 0"),
            "counts_out overlaps a 4-byte column": (lambda: call([good[0], (big.data_ptr(), F32, 0)],
                                                                 o=[None, None, big.data_ptr() + 8 * ((4 * n - 1) // 8)]),
                                                    "column 1"),
        }
        for what, (fn, word) in cases.items():
            assert fn() == ERR_ARG, what
            assert word in Lb.lsb_last_error(ctx).decode(), (what, Lb.lsb_last_error(ctx).decode())
        st = L.Stats()
        assert Lb.lsb_unique_device(ctx, cols(*good), 2, 0, None, None, None, n, ctypes.byref(u), None, ctypes.byref(st)) == 0
        want = U.reference([R.special_mix(n, "int64", seed=13), R.special_mix(n, "float32", seed=12)],
                           ["int64", "float32"], [False, True])
        assert u.value == len(want[0]) and st.passes == 6 and st.kernel_launches > 0
        assert call(good, uf=1) == 0
        want = U.reference([R.special_mix(n, "int64", seed=13), R.special_mix(n, "float32", seed=12)],
                           ["int64", "float32"], [False, True], consecutive=True)
        assert u.value == len(want[0]) and np.array_equal(outs[1].cpu().numpy(), want[1])
    for flags in (I64, F64, DESC):  # the order comes from the columns only
        with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
            assert s._L.lsb_unique_device(s._ctx, cols(*good), 2, 0, *ptrs, n, ctypes.byref(u), None, None) == ERR_ARG
            assert b"key-order" in s._L.lsb_last_error(s._ctx)
    with lsb.DistributedSorter(2 * n, world_size=2, world_rank=0) as s:  # one GPU only, refused before the comm state
        assert s._L.lsb_unique_device(s._ctx, cols(*good), 2, 0, *ptrs, n, ctypes.byref(u), None, None) == ERR_ARG
        assert b"one GPU" in s._L.lsb_last_error(s._ctx)
    with lsb.DistributedSorter(0, ranks=1) as s:  # count 0: no device pointer is looked at
        st = L.Stats()
        for uf, passes in ((0, 4 + 2), (1, 0)):
            u.value = -1
            assert s._L.lsb_unique_device(s._ctx, cols((None, 0, F64), (12345, F32, DESC)), 2, uf, 8, 16, 24, 0,
                                          ctypes.byref(u), None, ctypes.byref(st)) == 0
            assert u.value == 0 and st.passes == passes and st.elements == 0


def test_python_refusals():
    n = 1000
    x = torch.zeros(n, dtype=torch.int64, device="cuda")
    with lsb.DistributedSorter(n, ranks=1) as s:
        for bad in (dict(index_out=torch.zeros(n, dtype=torch.float64, device="cuda")),
                    dict(counts_out=torch.zeros(n, dtype=torch.int32, device="cuda")), dict(inverse_out=[0] * n),
                    dict(consecutive=1)):
            with pytest.raises(TypeError):
                s.unique_device([x], **bad)
        for bad in (dict(index_out=torch.zeros(n - 1, dtype=torch.int64, device="cuda")),
                    dict(inverse_out=torch.zeros(n, dtype=torch.int64))):
            with pytest.raises(ValueError):
                s.unique_device([x], **bad)
        with pytest.raises(ValueError):
            s.unique_device([x[1:]])
        with pytest.raises(TypeError):
            s.unique_device(x)
        index, inverse, counts, u, _ = s.unique_device([x], index_out=False, inverse_out=False, counts_out=False)
        assert (index, inverse, counts, u) == (None, None, None, 1)


# ---- 6. lsb.unique / lsb.unique_consecutive against torch and numpy ------------------------------------------------------
DTYPES = [torch.uint64, torch.int64, torch.float64, torch.uint32, torch.int32, torch.float32, torch.uint16, torch.int16,
          torch.float16, torch.bfloat16]


def _values(shape, dtype, k, seed):
    """NaN-free values of the dtype with few distinct ones (no -0.0, whose representative torch picks its own way)"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randint(0, k, shape, device="cuda", generator=g).to(torch.float32).mul(1.5).sub(3).round().to(dtype) \
        if dtype.is_floating_point else torch.randint(0, k, shape, device="cuda", generator=g).sub(k // 2 if dtype.is_signed else 0).to(dtype)


def _take(x, index):
    """x[index] through a signed view of x's width: torch indexes no unsigned CUDA tensor wider than a byte"""
    return x.view({8: torch.int64, 4: torch.int32, 2: torch.int16}[x.element_size()])[index].view(x.dtype)


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(-1).view(torch.uint8) if a.numel() else a,
                                                                        b.view(-1).view(torch.uint8) if b.numel() else b)


@pytest.mark.parametrize("dtype", DTYPES)
def test_against_torch(dtype):
    torch_has = dtype not in (torch.uint64, torch.uint32, torch.uint16)  # torch.unique's CUDA kernels lack these
    for shape, dim in [((100003,), None), ((57, 31, 3), None), ((9, 4, 5), 0), ((4, 9, 5), 1), ((4, 5, 9), 2),
                       ((4, 5, 9), -1), ((5000, 2), 0)]:
        x = _values(shape, dtype, 4 if dim is not None else 300, seed=len(shape) + (dim or 0))
        if dim is not None:
            x.select(dim, 1).copy_(x.select(dim, 0))  # two equal slices at least
        before = x.clone()
        got = lsb.unique(x, sorted=True, return_inverse=True, return_counts=True, dim=dim)
        cons = lsb.unique_consecutive(x, return_inverse=True, return_counts=True, dim=dim)
        assert _same(x, before)
        if torch_has:
            want = torch.unique(x, sorted=True, return_inverse=True, return_counts=True, dim=dim)
            assert all(_same(a, b) for a, b in zip(got, want)), (shape, dim)
            want = torch.unique_consecutive(x, return_inverse=True, return_counts=True, dim=dim)
            assert all(_same(a, b) for a, b in zip(cons, want)), (shape, dim)
        else:  # against the same values widened to int64, which keep the order
            wide = torch.unique(x.to(torch.int64), sorted=True, return_inverse=True, return_counts=True, dim=dim)
            assert torch.equal(got[0].to(torch.int64), wide[0]) and all(_same(a, b) for a, b in zip(got[1:], wide[1:]))
    # the plain forms and return_index
    x = _values((5000,), dtype, 50, seed=11)
    v = lsb.unique(x)
    assert isinstance(v, torch.Tensor) and torch.equal(v, lsb.unique(x, sorted=False))
    v2, index, inverse = lsb.unique(x, return_index=True, return_inverse=True)
    assert _same(v, v2) and _same(_take(x, index), v) and _same(_take(v, inverse), x)
    first = torch.full((len(v),), len(x), dtype=torch.int64, device="cuda")
    assert torch.equal(first.scatter_reduce(0, inverse, torch.arange(len(x), device="cuda"), "amin"), index)
    assert isinstance(lsb.unique_consecutive(x), torch.Tensor)


def test_scalar_and_empty():
    for dtype in (torch.int64, torch.float32, torch.int16):
        t = torch.tensor(3, device="cuda").to(dtype)
        got = lsb.unique(t, return_inverse=True, return_counts=True)
        assert [tuple(a.shape) for a in got] == [(1,), (), (1,)] and got[0].item() == 3 and got[2].item() == 1
        got = lsb.unique_consecutive(t, return_inverse=True, return_counts=True)
        assert [tuple(a.shape) for a in got] == [(1,), (), (1,)]
        for shape, dim in [((0,), None), ((2, 0), None), ((0, 3), 0), ((3, 0), 1)]:
            x = torch.zeros(shape, device="cuda").to(dtype)
            for fn, ref in ((lsb.unique, torch.unique), (lsb.unique_consecutive, torch.unique_consecutive)):
                got = fn(x, return_inverse=True, return_counts=True, dim=dim)
                want = ref(x.cpu(), return_inverse=True, return_counts=True, dim=dim)
                assert [(tuple(a.shape), a.dtype) for a in got] == [(tuple(a.shape), a.dtype) for a in want], (shape, dim)
                assert all(a.is_cuda for a in got)


def test_nans_as_numpy():
    """NaNs of both signs and payloads are one value, -0.0 == +0.0: numpy's equal_nan=True, not torch (which counts
    every NaN apart); values keep the bits of the first occurrence"""
    n = 200003
    for name in ("float64", "float32", "float16"):
        bits = R.special_mix(n, name, seed=5)
        x = R.to_device(torch, bits, name)
        v, index, inverse, counts = lsb.unique(x, return_index=True, return_inverse=True, return_counts=True)
        typed = R.typed(bits, name)
        wv, wi, winv, wc = np.unique(typed, return_index=True, return_inverse=True, return_counts=True, equal_nan=True)
        assert np.array_equal(index.cpu().numpy(), wi) and np.array_equal(inverse.cpu().numpy(), winv.reshape(-1))
        assert np.array_equal(counts.cpu().numpy(), wc)
        assert np.array_equal(v.cpu().numpy().view(bits.dtype), bits[wi])
        assert int(np.isnan(typed).any()) == int(torch.isnan(v).sum())
