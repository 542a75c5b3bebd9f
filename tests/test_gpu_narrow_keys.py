"""Narrow keys (uint32, int32, float32, uint16, int16, float16, bfloat16) on the GPU: lsb_sort_device_typed,
lsb_sort_segments_device_typed, a sorter made with key_dtype, and the torch.sort / torch.argsort drop-ins -- needs a
B200.

Every result is compared bit for bit (keys as their bit patterns, so NaN payloads and -0.0 count) with numpy's stable
argsort of the typed values (tests/narrow_keys.py; bfloat16 through its exact float32 widening) and, where torch sorts
the dtype on CUDA and there are no NaNs, with torch.sort(stable=True).
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import narrow_keys as NK  # noqa: E402
import patterns as P  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from test_gpu_patterns import _expected_skips  # noqa: E402

TL, OP, NS, DESC = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP, L.FLAG_DESCENDING
SHAPES = [0, NS, TL, OP, OP | NS, TL | OP]
SIZES = [P.PART_TILE + 1, P.SUPERTILE - 1, P.SUPERTILE + 1, (1 << 20) + 7]
ERR_ARG = -1


def _dt(name):
    return NK.torch_dtype(torch, name)


def _torch_check(kt, descending, got_k, got_v, dim=-1):
    """torch.sort(stable=True) agrees bit for bit where it sorts the dtype on CUDA and there are no NaNs"""
    if kt.is_floating_point() and bool(torch.isnan(kt).any()):
        return
    try:
        tk, ti = torch.sort(kt, dim=dim, stable=True, descending=descending)
    except (RuntimeError, NotImplementedError):
        return  # no CUDA sort of this dtype in this torch
    if got_k is not None:
        w = {8: torch.int64, 4: torch.int32, 2: torch.int16}[kt.element_size()]
        assert torch.equal(tk.view(w), got_k.view(w))
    assert torch.equal(ti, got_v)


def _check(bits, name, descending=False, flags=0, radix=16, vals=None, outputs="kv", sorter=None):
    """sort `bits` as keys of type `name` through a sorter made with key_dtype; returns (keys_out, vals_out, stats)"""
    n = len(bits)
    kt = NK.to_device(torch, bits, name)
    k_in = kt.clone()
    s = sorter or lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags | (DESC if descending else 0),
                                        key_dtype=_dt(name))
    try:
        k, v, st = s.sort_device(kt, vals, keys_out=None if "k" in outputs else False,
                                 vals_out=None if "v" in outputs else False)
        perm = NK.argsort(bits, name, descending)
        what = (name, descending, flags, radix, n)
        if "k" in outputs:
            assert k.dtype == kt.dtype and np.array_equal(NK.bits_of(torch, k), bits[perm]), what
        else:
            assert k is None
        if "v" in outputs:
            want = perm if vals is None else vals.view(torch.int64).cpu().numpy()[perm]
            assert np.array_equal(v.view(torch.int64).cpu().numpy(), want), what
        else:
            assert v is None
        if outputs == "kv" and vals is None:
            _torch_check(kt, descending, k, v)
        assert np.array_equal(NK.bits_of(torch, kt), NK.bits_of(torch, k_in))  # input untouched
        assert st.passes == -(-NK.BITS[name] // s.radix_bits), what
        return k, v, st
    finally:
        if sorter is None:
            s.close()


# ---- 1. every type x order x pass shape x size --------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("name", NK.NAMES)
def test_types_shapes_sizes(name, descending, n):
    bits = NK.special_mix(n, name, seed=n)
    for flags in SHAPES:
        _check(bits, name, descending, flags)


@pytest.mark.parametrize("n", [0, 1, 31, 33])
@pytest.mark.parametrize("name", NK.NAMES)
def test_tiny_sizes(name, n):
    bits = NK.special_mix(n, name, seed=3)
    for descending in (False, True):
        for flags in SHAPES:
            _check(bits, name, descending, flags)


@pytest.mark.parametrize("radix", [8, 11, 13, 16])
@pytest.mark.parametrize("name", NK.NAMES)
def test_radix_widths(name, radix):
    """radix 13 does not divide 32 or 16: the last digit is clamped to the key (13, 13, 6 / 13, 3 bits)"""
    bits = NK.special_mix(P.SUPERTILE + 1, name, seed=radix)
    for descending in (False, True):
        for flags in (0, TL, OP, TL | OP):
            _, _, st = _check(bits, name, descending, flags, radix=radix)
            assert st.passes == -(-NK.BITS[name] // radix)


# ---- 2. skipped passes --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["uint32", "int16", "float32"])
def test_skipped_steps(name):
    """keys with constant bytes skip their steps; all-equal keys skip every step and never leave the first shard"""
    w = NK.BITS[name]
    n = P.SUPERTILE + 1
    rng = np.random.default_rng(21)
    low = rng.integers(0, 256, n, dtype=np.uint64)
    # only the low byte of the order key varies: k (uint32), k ^ 0x8000 (int16), k ^ 2^31 (positive float32 0x3F8000xx)
    base = {"uint32": 0x12345600, "int16": 0x8300, "float32": 0x3F800000}[name]
    bits = (np.uint64(base) | low).astype(NK.UINT[w])
    order = (bits.astype(np.uint64) ^ (np.uint64(1 << (w - 1)) if name != "uint32" else np.uint64(0)))
    for flags in (0, OP, TL, TL | OP, NS):
        _, _, st = _check(bits, name, False, flags)
        assert st.skipped == _expected_skips(order, flags, passes=range(-(-w // 16))), (name, flags)
    same = np.full(10007, bits[0], dtype=NK.UINT[w])
    for flags in (0, OP, TL):
        _, v, st = _check(same, name, True, flags)
        assert st.skipped == (w // 8 if flags == 0 else w // 16) and np.array_equal(v.cpu().numpy(), np.arange(10007))


# ---- 3. values and outputs ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("outputs", ["kv", "k", "v"])
@pytest.mark.parametrize("vals", ["index", "int64", "float64"])
@pytest.mark.parametrize("name", ["float32", "bfloat16", "int16"])
def test_vals_and_outputs(name, vals, outputs):
    n = P.SUPERTILE + 1
    bits = NK.special_mix(n, name, seed=5)
    rng = np.random.default_rng(6)
    v = None
    if vals == "int64":
        v = torch.from_numpy(rng.integers(-(1 << 63), (1 << 63) - 1, n, dtype=np.int64)).cuda()
    elif vals == "float64":
        v = torch.from_numpy(rng.standard_normal(n)).cuda()
    for flags in (0, OP, TL):
        _check(bits, name, flags == OP, flags, vals=v, outputs=outputs)


@pytest.mark.parametrize("name", NK.NAMES)
def test_unaligned_views_and_in_place(name):
    """keys need alignment to their own width only: t[1:] of a 2- or 4-byte tensor; outputs may be the inputs"""
    n = (1 << 20) + 7
    bits = NK.special_mix(n + 1, name, seed=7)
    base = NK.to_device(torch, bits, name)
    keys = base[1:]
    assert keys.data_ptr() % 8 != 0
    vals = (torch.arange(n + 3, dtype=torch.int64, device="cuda") * 3)[3:]
    ko = torch.empty(n + 1, dtype=keys.dtype, device="cuda")[1:]
    vo = torch.empty(n + 1, dtype=torch.int64, device="cuda")[1:]
    perm = NK.argsort(bits[1:], name)
    with lsb.DistributedSorter(n, ranks=1, key_dtype=_dt(name)) as s:
        k, v, _ = s.sort_device(keys, vals, keys_out=ko, vals_out=vo)
        assert k is ko and v is vo
        assert np.array_equal(NK.bits_of(torch, k), bits[1:][perm])
        assert np.array_equal(v.cpu().numpy(), (np.arange(3, n + 3) * 3)[perm])
        k, v, _ = s.sort_device(keys, keys_out=keys)  # in place
        assert k is keys and np.array_equal(NK.bits_of(torch, base[1:]), bits[1:][perm])
        assert np.array_equal(v.cpu().numpy(), perm)
        assert NK.bits_of(torch, base[:1])[0] == bits[0]


# ---- 4. a reused sorter and stream ordering ------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, OP, TL])
def test_reused_sorter(flags):
    n = P.SUPERTILE + 1
    with lsb.DistributedSorter(n, ranks=1, flags=flags | DESC, key_dtype=torch.float16) as s:
        for seed in range(4):
            bits = NK.special_mix(n, "float16", seed=100 + seed) if seed != 2 else np.full(n, 0x7E12, dtype=np.uint16)
            k, v, _ = _check(bits, "float16", True, sorter=s)
            k2, v2, _ = _check(bits, "float16", True, flags)
            assert torch.equal(k.view(torch.int16), k2.view(torch.int16)) and torch.equal(v, v2)


@pytest.mark.parametrize("flags", [0, OP, TL])
def test_narrow_calls_leave_the_context_plan(flags):
    """Typed calls sort by their own plan (a float32 key at radix 13 is digits of 13, 13 and 6 bits, ascending in the
    packed word) and leave the context's (five digits of a 64-bit word, descending): interleaved on one sorter, every
    call returns what it returns on a fresh sorter."""
    n, radix = P.SUPERTILE + 1, 13
    rng = np.random.default_rng(18)
    bits = NK.special_mix(n, "float32", seed=18)
    kt = NK.to_device(torch, bits, "float32")
    offsets = torch.from_numpy(np.concatenate([[0], np.sort(rng.integers(0, n, 99)), [n]]).astype(np.int64)).cuda()
    recs = np.empty(n, dtype=L.ELT)
    recs["key"] = KO.special_mix(n, seed=18)
    recs["val"] = np.arange(n)

    def typed(s):
        k, v, st = s.sort_device(kt)
        return NK.bits_of(torch, k), v.cpu().numpy(), st.passes

    def segments(s):
        k, v, st = s.sort_segments(kt, offsets)
        return NK.bits_of(torch, k), v.cpu().numpy(), st.passes

    def records(s):
        s.upload(recs)
        st = s.my_sort()
        return s.download().view(np.uint64), st.passes

    def plan(s):
        return s.num_passes(), [s.digit_bits(d) for d in range(s.num_passes())]

    def sorter():
        return lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags | DESC, key_dtype=torch.float32)

    with sorter() as s:
        for call in [typed, records, segments, plan, records, typed, segments, records, plan]:
            got = call(s)
            with sorter() as fresh:
                want = call(fresh)
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), call.__name__
        assert plan(s) == (5, [13, 13, 13, 13, 12])
        k, v, passes = typed(s)
        perm = NK.argsort(bits, "float32", True)
        assert np.array_equal(k, bits[perm]) and np.array_equal(v, perm) and passes == 3


def test_waits_for_the_callers_stream():
    n = (1 << 20) + 7
    bits = NK.special_mix(n, "float32", seed=11)
    new = NK.to_device(torch, bits, "float32")
    keys = torch.zeros(n, dtype=torch.float32, device="cuda")
    side = torch.cuda.Stream()
    with lsb.DistributedSorter(n, ranks=1, key_dtype=torch.float32) as s:
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(100_000_000)  # tens of ms on the side stream before the keys are written
            keys.copy_(new)
        k, v, _ = s.sort_device(keys, stream=side)  # no synchronise in between
    perm = NK.argsort(bits, "float32")
    assert np.array_equal(NK.bits_of(torch, k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)


# ---- 5. the C entry points ------------------------------------------------------------------------------------------------
def test_c_level_refusals():
    n = 10007
    bits = NK.special_mix(n, "float32", seed=12)
    keys = NK.to_device(torch, bits, "float32")
    h16 = NK.to_device(torch, NK.special_mix(n, "bfloat16", seed=12), "bfloat16")
    out = torch.empty(3 * n, dtype=torch.int64, device="cuda")
    offsets = torch.tensor([0, n // 2, n], dtype=torch.int64, device="cuda")
    with lsb.DistributedSorter(n, ranks=1) as s:
        Lb, ctx = s._L, s._ctx
        kp, hp, op = keys.data_ptr(), h16.data_ptr(), out.data_ptr()

        def call(kt, k, v, ko, vo):
            return Lb.lsb_sort_device_typed(ctx, kt, k, v, ko, vo, n, None, None)

        def call_seg(kt, k, v, ko, vo):
            return Lb.lsb_sort_segments_device_typed(ctx, kt, k, v, ko, vo, n, offsets.data_ptr(), 2, 0, None, None)

        F32, BF16 = NK.KEY_TYPE["float32"], NK.KEY_TYPE["bfloat16"]
        cases = {
            "unknown key_type 8": (8, kp, None, op, None),
            "unknown key_type 2^31": (1 << 31, kp, None, op, None),
            "misaligned 4-byte keys": (F32, kp + 2, None, op, None),
            "misaligned 2-byte keys": (BF16, hp + 1, None, op, None),
            "misaligned 4-byte keys_out": (F32, kp, None, op + 2, None),
            "misaligned vals_out": (F32, kp, None, None, op + 4),
            "keys_out overlaps vals_out by one 4-byte key": (F32, kp, None, op, op + (4 * n - 1) // 8 * 8),
            "keys_out overlaps vals_out by 2-byte keys": (BF16, hp, None, op, op + (2 * n - 1) // 8 * 8),
            "no outputs": (F32, kp, None, None, None),
            "the context's own shard": (F32, s.device_ptr(), None, op, None),
        }
        for what, args in cases.items():
            for fn in (call, call_seg):
                assert fn(*args) == ERR_ARG, what
                assert Lb.lsb_last_error(ctx).decode(), what
        # keys_out of 4 n bytes followed by vals_out at the next 8-byte boundary: the real widths do not overlap
        va = (4 * n + 7) // 8
        assert call(F32, kp, None, op, op + 8 * va) == 0
        perm = NK.argsort(bits, "float32")
        assert np.array_equal(out.view(torch.int32)[:n].cpu().numpy().view(np.uint32), bits[perm])
        assert np.array_equal(out[va:va + n].cpu().numpy(), perm)
    with lsb.DistributedSorter(n, ranks=1, flags=L.FLAG_KEY_F64) as s:  # a narrow type on an 8-byte-typed context
        for fn in ("lsb_sort_device_typed", "lsb_sort_segments_device_typed"):
            args = (s._ctx, F32, kp, None, op, None, n) + ((offsets.data_ptr(), 2, 0) if "segments" in fn else ()) + (None, None)
            assert getattr(s._L, fn)(*args) == ERR_ARG and b"narrow" in s._L.lsb_last_error(s._ctx)


@pytest.mark.parametrize("order", ["u64", "i64_desc", "f64"])
def test_key_context_through_the_typed_calls(order):
    """LSB_KEY_CONTEXT: lsb_sort_device_typed is lsb_sort_device and the segmented form is lsb_sort_segments_device"""
    korder = KO.ORDERS[order]
    n = P.SUPERTILE + 1
    bits = KO.special_mix(n, seed=13)
    keys = torch.from_numpy(bits.view(np.int64)).cuda()
    offsets = torch.tensor([0, 1000, 1000, n], dtype=torch.int64, device="cuda")
    outs = [torch.empty(2 * n, dtype=torch.int64, device="cuda") for _ in range(4)]
    with lsb.DistributedSorter(n, ranks=1, flags=korder) as s:
        p = [o.data_ptr() for o in outs]
        st = [L.Stats() for _ in range(4)]
        assert s._L.lsb_sort_device(s._ctx, keys.data_ptr(), None, p[0], p[0] + 8 * n, n, None, ctypes.byref(st[0])) == 0
        assert s._L.lsb_sort_device_typed(s._ctx, 0, keys.data_ptr(), None, p[1], p[1] + 8 * n, n, None,
                                          ctypes.byref(st[1])) == 0
        assert s._L.lsb_sort_segments_device(s._ctx, keys.data_ptr(), None, p[2], p[2] + 8 * n, n, offsets.data_ptr(), 3,
                                             0, None, ctypes.byref(st[2])) == 0
        assert s._L.lsb_sort_segments_device_typed(s._ctx, 0, keys.data_ptr(), None, p[3], p[3] + 8 * n, n,
                                                   offsets.data_ptr(), 3, 0, None, ctypes.byref(st[3])) == 0
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[2], outs[3])
    assert st[0].passes == st[1].passes == 4 and st[2].passes == st[3].passes == 5
    assert np.array_equal(outs[0][n:].cpu().numpy(), KO.argsort(bits, korder))


# ---- 6. segments and rows ------------------------------------------------------------------------------------------------
def _segment_reference(bits, name, offsets, descending):
    """global input indices of the stable sort by (segment, key)"""
    perm = np.empty(len(bits), dtype=np.int64)
    for a, b in zip(offsets[:-1], offsets[1:]):
        perm[a:b] = a + NK.argsort(bits[a:b], name, descending)
    return perm


@pytest.mark.parametrize("name", NK.NAMES)
def test_segments(name):
    n = (1 << 20) + 7
    bits = NK.special_mix(n, name, seed=15)
    rng = np.random.default_rng(16)
    off = np.concatenate([[0], np.sort(rng.integers(0, n, 999)), [n]]).astype(np.int64)
    off[5] = off[4]  # an empty segment
    offsets = torch.from_numpy(off).cuda()
    kt = NK.to_device(torch, bits, name)
    vals = torch.from_numpy(rng.standard_normal(n)).cuda()
    for descending in (False, True):
        perm = _segment_reference(bits, name, off, descending)
        seg = np.searchsorted(off, np.arange(n), side="right") - 1
        for flags in (0, OP, TL):
            with lsb.DistributedSorter(n, ranks=1, flags=flags | (DESC if descending else 0), key_dtype=_dt(name)) as s:
                k, v, st = s.sort_segments(kt, offsets)  # global index
                assert np.array_equal(NK.bits_of(torch, k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)
                assert st.passes == NK.BITS[name] // 16 + 1  # key passes + one pass of the 10-bit segment id
                _, v, _ = s.sort_segments(kt, offsets, local_index=True, keys_out=False)
                assert np.array_equal(v.cpu().numpy(), perm - off[seg])
                k, v, _ = s.sort_segments(kt, offsets, vals=vals)  # gathered
                assert np.array_equal(v.cpu().numpy(), vals.cpu().numpy()[perm])
                assert np.array_equal(NK.bits_of(torch, k), bits[perm])


def test_segments_skip_segment_digits():
    """3 segments at radix 16: one segment pass whose high sub-digit is constant and skipped; one segment: no retag"""
    n = P.SUPERTILE + 1
    bits = NK.special_mix(n, "int32", seed=17)
    kt = NK.to_device(torch, bits, "int32")
    for off in ([0, 100, 5000, n], [0, n]):
        offsets = torch.tensor(off, dtype=torch.int64, device="cuda")
        perm = _segment_reference(bits, "int32", np.array(off), False)
        with lsb.DistributedSorter(n, ranks=1, key_dtype=torch.int32) as s:
            k, v, st = s.sort_segments(kt, offsets)
        assert np.array_equal(NK.bits_of(torch, k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)
        assert st.passes == 2 + (len(off) > 2)
        order = NK.bits_of(torch, kt).astype(np.uint64) ^ np.uint64(1 << 31)
        assert st.skipped == _expected_skips(order, 0, passes=range(2)) + (1 if len(off) > 2 else 0)


# ---- 7. sort / argsort: torch.sort drop-ins -------------------------------------------------------------------------------
ALL_DTYPES = ["uint64", "int64", "float64"] + NK.NAMES


def _bits_any(n, name, seed):
    if name in NK.BITS:
        return NK.special_mix(n, name, seed=seed)
    return KO.special_mix(n, seed=seed)


def _tensor_any(bits, name, shape):
    if name in NK.BITS:
        return NK.to_device(torch, bits, name).view(shape)
    return torch.from_numpy(bits.view(np.int64)).cuda().view(getattr(torch, name)).view(shape)


def _np_bits(t):
    w = {8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()]
    return t.contiguous().view(w).cpu().numpy()


def _reference(bits, name, shape, dim, descending):
    if name in NK.BITS:
        return NK.argsort(bits.reshape(shape), name, descending, axis=dim)
    x = np.moveaxis(KO.typed(bits, KO.ORDERS[{"uint64": "u64", "int64": "i64", "float64": "f64"}[name]]).reshape(shape), dim, -1)
    w = x.shape[-1]
    p = w - 1 - np.argsort(x[..., ::-1], axis=-1, kind="stable")[..., ::-1] if descending else np.argsort(x, axis=-1, kind="stable")
    return np.moveaxis(p, -1, dim)


@pytest.mark.parametrize("name", ALL_DTYPES)
def test_sort_and_argsort(name):
    for shape in [(), (0,), (1,), (1000,), (3, 0, 2), (33, 47), (1, 777), (5, 1), (4, 9, 300)]:
        for dim in sorted({d for d in (0, len(shape) // 2, -1) if len(shape) or d in (0, -1)}):
            for descending in (False, True):
                n = int(np.prod(shape)) if shape else 1
                bits = _bits_any(n, name, seed=4 * n + dim % 4)
                x = _tensor_any(bits, name, shape)
                r = lsb.sort(x, dim=dim, descending=descending)
                assert isinstance(r, torch.return_types.sort)
                values, indices = r
                assert values.shape == x.shape and indices.shape == x.shape and indices.dtype == torch.int64
                assert values.dtype == x.dtype
                what = (name, shape, dim, descending)
                if len(shape) == 0:
                    assert indices.item() == 0 and np.array_equal(_np_bits(values), _np_bits(x)), what
                    continue
                perm = _reference(bits, name, shape, dim, descending)
                assert np.array_equal(indices.cpu().numpy(), perm), what
                want = np.take_along_axis(_np_bits(x), perm, axis=dim)
                assert np.array_equal(_np_bits(values), want), what
                assert torch.equal(lsb.argsort(x, dim=dim, descending=descending, stable=True), indices), what
                _torch_check(x, descending, values, indices, dim=dim)


@pytest.mark.parametrize("name", ["float32", "bfloat16", "int64"])
def test_sort_transposed_and_strided_inputs(name):
    bits = _bits_any(300 * 77, name, seed=19)
    base = _tensor_any(bits, name, (300, 77))
    for x in (base.t(), base[::2, 1::3], base.t()[5]):
        assert not x.is_contiguous()
        xb = _np_bits(x)
        for dim in range(x.dim()):
            values, indices = lsb.sort(x, dim=dim, descending=True)
            perm = _reference(xb.reshape(-1).view(np.uint64 if x.element_size() == 8 else NK.UINT[8 * x.element_size()]),
                              name, x.shape, dim, True)
            assert np.array_equal(indices.cpu().numpy(), perm)
            assert np.array_equal(_np_bits(values), np.take_along_axis(xb, perm, axis=dim))


def test_sort_refuses_bad_dims():
    x = torch.zeros(3, 4, dtype=torch.float32, device="cuda")
    for dim in (2, -3, 1.0, None, True):
        with pytest.raises(ValueError):
            lsb.sort(x, dim=dim)
    with pytest.raises(ValueError):
        lsb.argsort(torch.zeros((), dtype=torch.bfloat16, device="cuda"), dim=1)
    with pytest.raises(TypeError):
        lsb.sort(torch.zeros(4, dtype=torch.int8, device="cuda"))
    with lsb.DistributedSorter(16, ranks=1, key_dtype=torch.float32) as s:
        with pytest.raises(TypeError):
            s.sort_device(torch.zeros(16, dtype=torch.float32, device="cuda"),
                          keys_out=torch.zeros(16, dtype=torch.int32, device="cuda"))
