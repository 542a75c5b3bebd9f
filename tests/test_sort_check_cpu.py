"""The independent sort checker (tests/sort_check.py) on the CPU: its order key against key_orders.order_key, its verdict
against np.lexsort on random small cases, every kind of wrong output it must report, and the bit layouts of the large
GPU cases (tests/test_gpu_large.py) -- so that editing their sizes cannot silently weaken them.  No GPU needed."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import key_orders as KO  # noqa: E402
import sort_check as C  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from test_segments_cpu import ragged_offsets, segment_ids  # noqa: E402

ORDER_NAMES = sorted(KO.ORDERS)


def _t(bits):
    return torch.from_numpy(np.ascontiguousarray(bits, dtype=np.uint64).view(np.int64))


def _reference(bits, off, korder):
    return np.lexsort((KO.order_key(bits, korder), segment_ids(off, len(bits))))


def _keys(rng, n, korder):
    """special values for f64, heavy ties otherwise"""
    if korder & KO.F64:
        return KO.special_mix(n, seed=int(rng.integers(1 << 30)))
    return rng.integers(0, 8, n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)  # both signs as int64


# ---- 1. the order key ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDER_NAMES)
def test_order_key_equals_key_orders(order):
    korder = KO.ORDERS[order]
    rng = np.random.default_rng(1)
    bits = np.concatenate([KO.SPECIAL_BITS, rng.integers(0, 1 << 64, 10000, dtype=np.uint64, endpoint=False)])
    want = (KO.order_key(bits, korder) ^ KO.TOP).view(np.int64)  # the same order, shifted into int64
    assert np.array_equal(C.order_key(_t(bits), korder).numpy(), want)
    assert C.SPECIAL_BITS == [int(b) for b in KO.SPECIAL_BITS.view(np.int64)]


def test_splitmix64_is_the_reference_generator():
    x = np.arange(1000, dtype=np.uint64) + np.uint64(5 << 40)
    with np.errstate(over="ignore"):
        z = (x + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    assert np.array_equal(C.splitmix64(_t(x)).numpy().view(np.uint64), z)
    assert int(C.splitmix64(torch.zeros(1, dtype=torch.int64))[0]) == C._s64(0xE220A8397B1DCDAF)  # splitmix64(seed 0)


def test_key_makers():
    n = (1 << 16) + 3
    a, b = C.uniform_keys(n, "cpu", seed=1), C.uniform_keys(n, "cpu", seed=2)
    assert not torch.equal(a, b) and torch.equal(a, C.uniform_keys(n, "cpu", seed=1))
    assert len(torch.unique(a)) == n and (a < 0).any()  # all 64 bits used
    h = C.heavy_hitter_keys(n, "cpu")
    cold = int((h != C.HOT_KEY).sum())
    assert 0 < cold < 2 * n >> C.COLD_SHIFT
    big = (1 << 31) + (1 << 20) + 7  # the hot key of the large GPU cases: more than 2^31 elements even with 10 % more
    assert big - (big >> C.COLD_SHIFT) * 11 // 10 > 1 << 31  # cold keys than expected (hundreds of standard deviations)
    d = C.special_doubles(n, "cpu").numpy().view(np.uint64)
    special = np.isin(d, KO.SPECIAL_BITS)
    assert 0.4 < special.mean() < 0.6 and set(d[special]) == set(KO.SPECIAL_BITS)
    normal = np.abs(d[~special].view(np.float64))
    assert (normal >= 2.0 ** -10).all() and (normal < 2.0 ** 11).all()
    off = C.ragged_offsets(n, 1001, "cpu", seed=3, long_segment=n - 500).numpy()
    assert len(off) == 1002 and off[0] == 0 and off[-1] == n and (np.diff(off) >= 0).all()
    assert off[1] == 0 and off[-2] == n and np.diff(off).max() >= n - 500 and (np.diff(off) == 0).sum() > 100


# ---- 2. the verdict against np.lexsort on random small cases -----------------------------------------------------------
def _segmentations(rng, n):
    yield None
    yield ragged_offsets(rng, n, 7)
    yield np.array([0, 0, 0, n // 3, n // 3, n, n, n], dtype=np.int64)  # empty first, inside and last
    yield np.arange(n + 1, dtype=np.int64) if n else np.array([0, 0])   # length 1


@pytest.mark.parametrize("chunk", [1, 5, 1 << 27])
@pytest.mark.parametrize("order", ORDER_NAMES)
def test_passes_exactly_the_stable_sort(order, chunk):
    korder = KO.ORDERS[order]
    rng = np.random.default_rng(KO.ORDERS[order] + chunk)
    for n in (0, 1, 2, 37, 300):
        bits = _keys(rng, n, korder)
        for off in _segmentations(rng, n):
            segs = np.array([0, n], dtype=np.int64) if off is None else off
            perm = _reference(bits, segs, korder)
            ot = None if off is None else torch.from_numpy(off)
            kin, kout = _t(bits), _t(bits[perm])
            assert C.check_sort(kin, kout, torch.from_numpy(perm), korder, ot, chunk=chunk) is None, (n, off)
            local = perm - segs[segment_ids(segs, n)[perm]]
            assert C.check_sort(kin, kout, C.LocalIndex(torch.from_numpy(local), torch.from_numpy(segs)), korder, ot,
                                chunk=chunk) is None
            for dtype in (torch.int64, torch.float64):
                vals = C.gather_vals(n, "cpu", dtype)
                assert C.check_sort(kin, kout, C.GatheredVals(vals[torch.from_numpy(perm)]), korder, ot, chunk=chunk) is None
            # any other permutation is reported, with the keys it gathers
            for _ in range(3):
                other = rng.permutation(n)
                if not np.array_equal(other, perm):
                    assert C.check_sort(kin, _t(bits[other]), torch.from_numpy(other), korder, ot, chunk=chunk)


def test_global_index_is_lexsort_order():
    """the stable sort is unique: an output passes only when it is np.lexsort's"""
    rng = np.random.default_rng(7)
    n = 64
    bits = rng.integers(0, 3, n, dtype=np.uint64)  # many equal keys: only the stable order passes
    off = np.array([0, 20, 20, 64], dtype=np.int64)
    perm = _reference(bits, off, 0)
    passed = 0
    for t in range(2000):
        cand = perm.copy()
        a, b = rng.integers(0, n, 2)
        cand[a], cand[b] = cand[b], cand[a]
        ok = C.check_sort(_t(bits), _t(bits[cand]), torch.from_numpy(cand), 0, torch.from_numpy(off)) is None
        assert ok == np.array_equal(cand, perm)
        passed += ok
    assert passed > 0


# ---- 3. mutations of a correct output ------------------------------------------------------------------------------------
N = 1000


def _case(korder=KO.F64, seed=0):
    rng = np.random.default_rng(seed)
    bits = KO.special_mix(N, seed=seed)
    off = ragged_offsets(rng, N, 9)
    perm = _reference(bits, off, korder)
    return bits, off, perm


def _fails(bits, kout_bits, idx, korder, off, want):
    msg = C.check_sort(_t(bits), _t(kout_bits), idx, korder, None if off is None else torch.from_numpy(off), chunk=128)
    assert msg is not None and msg.startswith(want), msg
    return msg


def _pair(bits, perm, off, korder, equal):
    """adjacent output positions j, j + 1 in one segment with equal (or unequal) order keys"""
    ok = KO.order_key(bits[perm], korder)
    seg = segment_ids(off, N)
    same = (seg[:-1] == seg[1:]) & ((ok[:-1] == ok[1:]) == equal)
    return int(np.flatnonzero(same)[len(np.flatnonzero(same)) // 2])


@pytest.mark.parametrize("korder", [KO.F64, KO.F64 | KO.DESC])
def test_stability_break(korder):
    bits, off, perm = _case(korder)
    j = _pair(bits, perm, off, korder, equal=True)
    bad = perm.copy()
    bad[j], bad[j + 1] = bad[j + 1], bad[j]
    msg = _fails(bits, bits[bad], torch.from_numpy(bad), korder, off, "check 4")
    assert f"from position {j} to {j + 1}" in msg and f">{j:>11}" in msg


def test_unequal_keys_swapped():
    bits, off, perm = _case()
    j = _pair(bits, perm, off, KO.F64, equal=False)
    bad = perm.copy()
    bad[j], bad[j + 1] = bad[j + 1], bad[j]
    _fails(bits, bits[bad], torch.from_numpy(bad), KO.F64, off, "check 4")


def test_index_duplicated():
    bits, off, perm = _case()
    bad = perm.copy()
    bad[500] = bad[400]
    msg = _fails(bits, bits[bad], torch.from_numpy(bad), KO.F64, off, "check 2")
    assert f"input index {perm[500]} is missing" in msg and "position 500 repeats" in msg


@pytest.mark.parametrize("value", [N, N + 12345, 1 << 40, -1, -(1 << 63)])
def test_index_out_of_range(value):
    """reported before any gather or scatter through idx: on the CPU an out-of-range index raises IndexError, so a
    checker that indexed first would fail here rather than return the message (on the device it would assert)"""
    bits, off, perm = _case()
    bad = perm.copy()
    bad[321] = value
    msg = _fails(bits, bits[perm], torch.from_numpy(bad), KO.F64, off, "check 1")
    assert "position 321" in msg and "out of range" in msg


def test_nan_payload_bit_flipped():
    bits, off, perm = _case()
    out = bits[perm].copy()
    nan = np.flatnonzero((out << np.uint64(1)) > np.uint64(0x7FF << 53))
    j = int(nan[len(nan) // 2])
    out[j] ^= np.uint64(1 << 3)  # still a NaN, same order key: only the bits tell
    assert (KO.order_key(out, KO.F64) == KO.order_key(bits[perm], KO.F64)).all()
    assert f"keys_out[{j}]" in _fails(bits, out, torch.from_numpy(perm), KO.F64, off, "check 3")


def test_negative_zero_written_as_positive_zero():
    bits, off, perm = _case()
    out = bits[perm].copy()
    j = int(np.flatnonzero(out == np.uint64(1 << 63))[0])
    out[j] = 0
    assert f"keys_out[{j}]" in _fails(bits, out, torch.from_numpy(perm), KO.F64, off, "check 3")


def test_element_moved_across_a_segment_boundary():
    """the last elements of two adjacent segments trade places: every segment still holds rising keys and the
    output is a permutation, so only the segment check sees it"""
    rng = np.random.default_rng(3)
    bits = np.sort(rng.integers(0, 1 << 40, N, dtype=np.uint64))  # ascending input: the sort is the identity
    off = torch.tensor([0, 300, 700, N])
    perm = np.arange(N)
    assert C.check_sort(_t(bits), _t(bits), torch.from_numpy(perm), 0, off) is None
    moved = perm.copy()
    moved[299], moved[300] = 300, 299  # input 299 (segment 0's largest) first in segment 1, input 300 last in segment 0
    msg = C.check_sort(_t(bits), _t(bits[moved]), torch.from_numpy(moved), 0, off)
    assert msg.startswith("check 5") and "position 299" in msg


def test_local_index_off_by_one():
    bits, off, perm = _case()
    local = perm - off[segment_ids(off, N)[perm]]
    for j, d in ((0, 1), (N // 2, -1), (N - 1, 1)):
        bad = local.copy()
        bad[j] += d
        _fails(bits, bits[perm], C.LocalIndex(torch.from_numpy(bad), torch.from_numpy(off)), KO.F64, off, "check")


@pytest.mark.parametrize("dtype", [torch.int64, torch.float64])
def test_gathered_value_low_bit_flipped(dtype):
    bits, off, perm = _case()
    got = C.gather_vals(N, "cpu", dtype)[torch.from_numpy(perm)].clone()
    got.view(torch.int64)[N // 3] ^= 1
    msg = _fails(bits, bits[perm], C.GatheredVals(got), KO.F64, off, "check 1")
    assert f"position {N // 3}" in msg


def test_message_shows_the_neighbourhood():
    bits, off, perm = _case()
    bad = perm.copy()
    bad[10], bad[11] = bad[11], bad[10]
    msg = _fails(bits, bits[bad], torch.from_numpy(bad), KO.F64, off, "check")
    rows = msg.splitlines()[2:]
    assert len(rows) == 2 * C.CONTEXT + 1 and [int(r[1:12]) for r in rows] == list(range(10 - C.CONTEXT, 11 + C.CONTEXT))


# ---- 4. the layouts of the large GPU cases --------------------------------------------------------------------------------
def test_layouts_of_the_gpu_cases():
    import test_gpu_large as G
    for radix, n, S in G.LAYOUT_64:
        idxbits, segbits, segw, passes, fits = H.segsort_layout(n, S, radix)
        assert fits and segw + idxbits == 64, (radix, n, S)
        assert n - 1 >= 1 << (idxbits - 1)  # the index's top bit -- bit 63 of the retagged word -- is used
    for S in (G.BIG_SEGMENTS, G.BIG_SEGMENTS_GATHER):
        idxbits, _, segw, passes, fits = H.segsort_layout(G.BIG, S, 16)
        assert fits and segw + idxbits == 64 and idxbits == 32 and passes == 2
    idxbits, _, segw, _, fits = H.segsort_layout(G.BIG, G.REFUSED_SEGMENTS, G.REFUSED_RADIX)
    assert not fits and segw + idxbits == 65
    assert G.BIG - 1 >= 1 << 31 and G.ROWS * G.WIDTH - 1 >= 1 << 31
    idxbits, _, segw, _, fits = H.segsort_layout(G.ROWS * G.WIDTH, G.ROWS, 16)
    assert fits and idxbits == 32
    assert G.LONG_SEGMENT > 1 << 31
