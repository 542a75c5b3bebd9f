"""Device tensors in, device tensors out: lsb_sort_device, DistributedSorter.sort_device and sort_tensor -- needs a B200.

Every result is compared bit for bit (keys through .view(torch.int64), so NaN payloads and -0.0 count) with numpy's
stable argsort of the typed keys (tests/key_orders.py) and, for int64 keys and float64 keys without NaNs, with
torch.sort(stable=True).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import patterns as P  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from oracle import oracle as O  # noqa: E402
from test_gpu_key_order import _infs, _mixed, _nans, _zeros  # noqa: E402
from test_gpu_patterns import _expected_skips  # noqa: E402

TL, OP, NS = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP
SHAPES = [0, NS, TL, OP, OP | NS, TL | OP]
SIZES = [P.PART_TILE + 1, P.SUPERTILE - 1, P.SUPERTILE + 1, (1 << 20) + 7]
TORCH_DTYPE = {np.uint64: torch.uint64, np.int64: torch.int64, np.float64: torch.float64}
ERR_ARG = -1


def _dtype(korder):
    return TORCH_DTYPE[KO.DTYPES[korder & (KO.I64 | KO.F64)]]


def _dev(bits, dtype):
    """uint64 numpy bits -> a CUDA tensor of `dtype` holding the same bits"""
    return torch.from_numpy(np.ascontiguousarray(bits).view(np.int64)).cuda().view(dtype)


def _bits(t):
    return t.view(torch.int64).cpu().numpy().view(np.uint64)


def _torch_comparable(kt):
    """torch.sort sorts int64 and float64 keys on CUDA, but it does not keep a NaN's bits and does not put every NaN
    last, so the comparison with it is made on keys without NaNs (numpy's order is the reference for those)"""
    return kt.dtype == torch.int64 or (kt.dtype == torch.float64 and not bool(torch.isnan(kt).any()))


def _torch_sort_check(kt, korder, got_k, got_v):
    """torch.sort(stable=True[, descending=True]) agrees bit for bit"""
    if not _torch_comparable(kt):
        return
    tk, ti = torch.sort(kt, stable=True, descending=bool(korder & KO.DESC))
    assert torch.equal(tk.view(torch.int64), got_k.view(torch.int64))
    assert torch.equal(ti, got_v)


def _check(bits, korder, flags=0, radix=16, vals=None, outputs="kv", sorter=None):
    """sort `bits` read as the order's dtype through sort_device; returns (keys_out, vals_out, sorter stats)"""
    n = len(bits)
    kt = _dev(bits, _dtype(korder))
    k_in = kt.clone()
    v_in = None if vals is None else vals.clone()
    s = sorter or lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=korder | flags)
    try:
        k, v, st = s.sort_device(kt, vals, keys_out=None if "k" in outputs else False,
                                 vals_out=None if "v" in outputs else False)
        perm = KO.argsort(bits, korder)
        if "k" in outputs:
            assert k.dtype == kt.dtype and np.array_equal(_bits(k), bits[perm]), (korder, flags, radix, n)
        else:
            assert k is None
        if "v" in outputs:
            want_v = perm if vals is None else vals.view(torch.int64).cpu().numpy()[perm]
            assert v.dtype == (torch.int64 if vals is None else vals.dtype)
            assert np.array_equal(v.view(torch.int64).cpu().numpy(), want_v), (korder, flags, radix, n)
        else:
            assert v is None
        if outputs == "kv" and vals is None:
            _torch_sort_check(kt, korder, k, v)
            rec = np.empty(n, dtype=P.ELT)
            rec["key"], rec["val"] = bits, np.arange(n, dtype=np.uint64)
            vf = s.verify()  # the shard holds the sorted records, as after my_sort
            assert vf.order_violations == 0 and vf.elements == n and list(vf.checksum) == O.checksum(rec)
        assert torch.equal(kt.view(torch.int64), k_in.view(torch.int64))  # inputs untouched when outputs are separate
        if vals is not None:
            assert torch.equal(vals.view(torch.int64), v_in.view(torch.int64))
        return k, v, st
    finally:
        if sorter is None:
            s.close()


# ---- 1. every order x pass shape x size ----------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("order", list(KO.ORDERS))
def test_orders_shapes_sizes(order, n):
    bits = KO.special_mix(n, seed=n)
    for flags in SHAPES:
        _check(bits, KO.ORDERS[order], flags)


@pytest.mark.parametrize("n", [0, 1, 31, 33])
@pytest.mark.parametrize("order", list(KO.ORDERS))
def test_tiny_sizes(order, n):
    bits = KO.special_mix(n, seed=3) if n else np.zeros(0, dtype=np.uint64)
    for flags in SHAPES:
        _check(bits, KO.ORDERS[order], flags)


@pytest.mark.parametrize("radix", [8, 11])
@pytest.mark.parametrize("order", list(KO.ORDERS))
def test_radix_widths(order, radix):
    bits = _mixed(P.SUPERTILE + 1, 2)
    for flags in (0, TL, OP, TL | OP):
        _check(bits, KO.ORDERS[order], flags, radix=radix)


# ---- 2. special-value mixes and structured keys (skipped passes leave the result in the first shard) ------------------
@pytest.mark.parametrize("mix", ["zeros", "nans", "infs"])
@pytest.mark.parametrize("order", ["f64", "f64_desc"])
def test_f64_mixes(mix, order):
    n = P.SUPERTILE + 1
    bits = {"zeros": _zeros, "nans": _nans, "infs": _infs}[mix](np.random.default_rng([len(mix), n]), n)
    for flags in SHAPES:
        _check(bits, KO.ORDERS[order], flags)


@pytest.mark.parametrize("name", ["heavy_0.9", "ascending", "all_but_one_mid", "all_but_one_last"])
@pytest.mark.parametrize("order", ["u64", "i64_desc", "f64"])
def test_patterns(name, order):
    bits = P.make(name, P.SUPERTILE + 1)["key"].copy()
    for flags in SHAPES:
        _, _, st = _check(bits, KO.ORDERS[order], flags)
        assert st.skipped == _expected_skips(KO.order_key(bits, KO.ORDERS[order]), flags), (name, order, flags)


def test_all_passes_skipped():
    """every key equal: every step is skipped, the records never leave the first shard, and unpack reads them there"""
    bits = np.full(10007, 0x7FF8000000000123, dtype=np.uint64)
    for order in ("f64", "f64_desc", "u64"):
        _, v, st = _check(bits, KO.ORDERS[order])
        assert st.skipped == 8 and np.array_equal(v.cpu().numpy(), np.arange(len(bits)))


# ---- 3. values and outputs ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("outputs", ["kv", "k", "v"])
@pytest.mark.parametrize("vals", ["index", "int64", "float64"])
@pytest.mark.parametrize("order", ["u64", "i64", "f64_desc"])
def test_vals_and_outputs(order, vals, outputs):
    n = P.SUPERTILE + 1
    bits = KO.special_mix(n, seed=5)
    rng = np.random.default_rng(6)
    v = None
    if vals == "int64":
        v = torch.from_numpy(rng.integers(-(1 << 63), (1 << 63) - 1, n, dtype=np.int64)).cuda()
    elif vals == "float64":
        v = torch.from_numpy(rng.standard_normal(n)).cuda()
    for flags in (0, OP, TL):
        _check(bits, KO.ORDERS[order], flags, vals=v, outputs=outputs)


# ---- 4. 8-byte-aligned views and in-place calls -----------------------------------------------------------------------
@pytest.mark.parametrize("order", ["i64", "f64", "f64_desc"])
def test_unaligned_views(order):
    korder = KO.ORDERS[order]
    n = (1 << 20) + 7
    bits = KO.special_mix(n + 1, seed=7)
    base = _dev(bits, _dtype(korder))
    keys = base[1:]                                  # 8-byte but not 16-byte aligned
    assert keys.data_ptr() % 16 == 8
    vbase = torch.arange(n + 3, dtype=torch.int64, device="cuda") * 3
    vals = vbase[3:]
    ko = torch.empty(n + 1, dtype=keys.dtype, device="cuda")[1:]
    vo = torch.empty(n + 1, dtype=torch.int64, device="cuda")[1:]
    with lsb.DistributedSorter(n, ranks=1, flags=korder) as s:
        k, v, _ = s.sort_device(keys, vals, keys_out=ko, vals_out=vo)
    assert k is ko and v is vo
    perm = KO.argsort(bits[1:], korder)
    assert np.array_equal(_bits(k), bits[1:][perm])
    assert np.array_equal(v.cpu().numpy(), (np.arange(3, n + 3) * 3)[perm])


@pytest.mark.parametrize("vals", [False, True])
@pytest.mark.parametrize("order", ["u64", "i64_desc", "f64"])
def test_in_place(order, vals):
    korder = KO.ORDERS[order]
    n = P.SUPERTILE + 1
    bits = KO.special_mix(n, seed=8)
    keys = _dev(bits, _dtype(korder))
    v = torch.from_numpy(np.random.default_rng(9).standard_normal(n)).cuda() if vals else None
    v0 = None if v is None else v.clone()
    for flags in (0, OP):
        keys.copy_(_dev(bits, _dtype(korder)))
        if v is not None:
            v.copy_(v0)
        with lsb.DistributedSorter(n, ranks=1, flags=korder | flags) as s:
            k, vo, _ = s.sort_device(keys, v, keys_out=keys, vals_out=v if vals else None)
        perm = KO.argsort(bits, korder)
        assert k is keys and np.array_equal(_bits(keys), bits[perm])
        if vals:
            assert vo is v and torch.equal(v.view(torch.int64), v0[torch.from_numpy(np.ascontiguousarray(perm)).cuda()].view(torch.int64))
        else:
            assert np.array_equal(vo.cpu().numpy(), perm)


def test_keys_in_place_into_vals_input():
    """outputs may alias inputs in any combination, as long as the two outputs do not overlap"""
    n = 100003
    bits = KO.special_mix(n, seed=10)
    keys = _dev(bits, torch.float64)
    vals = torch.arange(n, dtype=torch.int64, device="cuda").view(torch.float64)
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64) as s:
        k, v, _ = s.sort_device(keys, vals, keys_out=vals, vals_out=keys)  # swapped
    perm = KO.argsort(bits, KO.F64)
    assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.view(torch.int64).cpu().numpy(), perm)


# ---- 5. a sorter reused for several calls ---------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, OP, TL])
def test_reused_sorter(flags):
    n = P.SUPERTILE + 1
    korder = KO.F64 | KO.DESC
    with lsb.DistributedSorter(n, ranks=1, flags=korder | flags) as s:
        for seed in range(4):
            bits = KO.special_mix(n, seed=100 + seed) if seed != 2 else np.full(n, 7, dtype=np.uint64)
            k, v, _ = _check(bits, korder, sorter=s)
            k2, v2, _ = _check(bits, korder, flags)  # a fresh sorter
            assert torch.equal(k.view(torch.int64), k2.view(torch.int64)) and torch.equal(v, v2)


# ---- 6. stream ordering ----------------------------------------------------------------------------------------------
def test_waits_for_the_callers_stream():
    n = (1 << 20) + 7
    bits = KO.special_mix(n, seed=11)
    new = _dev(bits, torch.float64)
    keys = torch.zeros(n, dtype=torch.float64, device="cuda")
    side = torch.cuda.Stream()
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64) as s:
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(100_000_000)  # tens of ms on the side stream before the keys are written
            keys.copy_(new)
        k, v, _ = s.sort_device(keys, stream=side)  # no synchronise in between
    perm = KO.argsort(bits, KO.F64)
    assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)


# ---- 7. the C entry point refuses bad pointers -------------------------------------------------------------------------
def test_c_level_refusals():
    n = 10007
    bits = KO.special_mix(n, seed=12)
    keys = _dev(bits, torch.int64)
    out = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    host = np.zeros(n, dtype=np.int64)
    pinned = L.PinnedBuffer(n)
    with lsb.DistributedSorter(n, ranks=1, flags=KO.I64) as s:
        Lb, ctx = s._L, s._ctx
        kp, op = keys.data_ptr(), out.data_ptr()

        def call(k, v, ko, vo, count=n):
            return Lb.lsb_sort_device(ctx, k, v, ko, vo, count, None, None)

        cases = {
            "host keys": (host.ctypes.data, None, op, None),
            "pinned keys": (pinned.array.ctypes.data, None, op, None),
            "host output": (kp, None, host.ctypes.data, None),
            "misaligned keys": (kp + 4, None, op, None),
            "misaligned vals": (kp, kp + 12, op, None),
            "misaligned output": (kp, None, op + 4, None),
            "overlapping outputs": (kp, None, op, op + 8 * (n // 2)),
            "same output twice": (kp, None, op, op),
            "no outputs": (kp, None, None, None),
            "no keys": (None, None, op, None),
            "the context's own shard": (s.device_ptr(), None, op, None),
        }
        for what, args in cases.items():
            rc = call(*args)
            assert rc == ERR_ARG, what
            assert Lb.lsb_last_error(ctx).decode(), what
        assert call(kp, None, op, None, count=n - 1) == ERR_ARG
        assert call(kp, None, op, None, count=n + 1) == ERR_ARG
        # the context is still usable, and the adjacent, non-overlapping halves of one buffer are accepted
        assert call(kp, None, op, op + 8 * n) == 0
        perm = KO.argsort(bits, KO.I64)
        assert np.array_equal(_bits(out[:n]), bits[perm]) and np.array_equal(out[n:].cpu().numpy(), perm)
    pinned.free()


# ---- 8. sort_tensor ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("dtype", [np.uint64, np.int64, np.float64])
def test_sort_tensor_equals_sort_pairs(dtype, descending):
    for n in (0, 1, 10007, P.SUPERTILE + 1):
        bits = _mixed(n, 13) if n else np.zeros(0, dtype=np.uint64)
        keys = bits.view(dtype)
        kt = _dev(bits, TORCH_DTYPE[dtype])
        k, v = lsb.sort_tensor(kt, descending=descending)
        pk, pv = lsb.sort_pairs(keys, descending=descending)
        assert k.dtype == kt.dtype and v.dtype == torch.int64
        assert np.array_equal(_bits(k), pk.view(np.uint64)) and np.array_equal(v.cpu().numpy(), pv), (dtype, n)
        if _torch_comparable(kt):
            tk, ti = torch.sort(kt, stable=True, descending=descending)
            assert torch.equal(tk.view(torch.int64), k.view(torch.int64)) and torch.equal(ti, v)
        vals = np.arange(n, dtype=np.float64) * 0.5
        k2, v2 = lsb.sort_tensor(kt, torch.from_numpy(vals).cuda(), descending=descending)
        pk2, pv2 = lsb.sort_pairs(keys, vals, descending=descending)
        assert v2.dtype == torch.float64 and np.array_equal(v2.cpu().numpy(), pv2)
        assert np.array_equal(_bits(k2), pk2.view(np.uint64))


def test_sort_tensor_non_contiguous_input():
    n = 50001
    bits = KO.special_mix(2 * n, seed=14)
    base = _dev(bits, torch.float64)
    k, v = lsb.sort_tensor(base[::2])
    perm = KO.argsort(bits[::2].copy(), KO.F64)
    assert np.array_equal(_bits(k), bits[::2][perm]) and np.array_equal(v.cpu().numpy(), perm)


def test_sort_device_rejects_other_gpu_and_cpu_tensors():
    n = 1000
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64) as s:
        with pytest.raises(ValueError):
            s.sort_device(torch.zeros(n, dtype=torch.float64))
        with pytest.raises(TypeError):
            s.sort_device(torch.zeros(n, dtype=torch.int64, device="cuda"))
        with pytest.raises(ValueError):
            s.sort_device(torch.zeros(n - 1, dtype=torch.float64, device="cuda"))
        if torch.cuda.device_count() > 1:
            with pytest.raises(ValueError):
                s.sort_device(torch.zeros(n, dtype=torch.float64, device="cuda:1"))
