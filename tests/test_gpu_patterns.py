"""Structured keys (tests/patterns.py) through every pass shape, bit for bit against the stable sort -- needs a B200.

The rest of the GPU suite sorts pcg64 keys, which almost never reach the paths that depend on the data: the spill of the
16-bit shared-memory digit counters, the rule that skips a pass whose digit is constant, parts of the virtual-rank pass
that are empty or 32 elements long, and the skewed inputs of the exchange kernel's fused next-digit count.  Every
expected value here comes from numpy (stable argsort, bincount, cumsum) or from the C oracle's single pass.
"""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import distributed_lsb_b200 as lsb  # noqa: E402
import patterns as P  # noqa: E402
from conftest import LIB_DEFAULT_TUNE, apply_session_tune  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from oracle import oracle as O  # noqa: E402

TL, OP, NS = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP
SHAPES = [0, NS, TL, OP, OP | NS, TL | OP]
# one partition tile plus one, the one-pass supertile minus and plus one, ragged
SIZES = [P.PART_TILE + 1, P.SUPERTILE - 1, P.SUPERTILE + 1, (1 << 20) + 7]

# every lsb_tune key at the library's built-in value (Tuning in csrc/lsbsort.cu)
LIB_DEFAULTS = {**P.TUNE_DEFAULTS, **LIB_DEFAULT_TUNE}


@pytest.fixture
def lib_tune():
    """lsb.tune for one test; afterwards every key is back at the built-in default, then the session's values"""
    try:
        yield lsb.tune
    finally:
        for k, v in LIB_DEFAULTS.items():
            lsb.tune(k, v)
        apply_session_tune()


@functools.lru_cache(maxsize=16)
def _case(name, n, vals="index"):
    a = P.make(name, n, vals)
    return a, P.reference(a)


def _sort(a, flags=0, radix=16):
    with lsb.DistributedSorter(len(a), radix_bits=radix, flags=flags) as s:
        s.upload(a)
        st = s.my_sort()
        return s.download(), st


def _assert_same(got, want, *ctx):
    g, w = got.view(np.uint64).reshape(-1, 2), want.view(np.uint64).reshape(-1, 2)
    if not np.array_equal(g, w):
        bad = np.flatnonzero((g != w).any(axis=1))
        i = int(bad[0])
        raise AssertionError(f"{ctx}: {len(bad)} records differ, first at {i}: got ({int(g[i, 0]):016x},{int(g[i, 1])}) "
                             f"want ({int(w[i, 0]):016x},{int(w[i, 1])})")


def _expected_skips(keys, flags, radix=16, passes=None):
    """steps a sort of `keys` skips: a stable step on a (sub-)digit that is constant over the array is the identity.
    The two-step shape decides per sub-digit (hostlogic.plan_pass), the others per digit."""
    if flags & NS or len(keys) == 0:
        return 0
    varying = int(np.bitwise_or.reduce(keys ^ keys[0]))  # the key bits that are not the same in every element

    def constant(shift, bits):
        return (varying >> shift) & ((1 << bits) - 1) == 0

    skips = 0
    for p in (range(H.num_passes(radix)) if passes is None else passes):
        shift, bits, lo, hi = H.plan_pass(radix, p, one_pass=bool(flags & OP))
        if flags & (TL | OP) or not lo:
            skips += constant(shift, bits)
        else:
            skips += constant(shift, lo) + constant(shift + lo, hi)
    return skips


def _shape(flags):
    return "+".join(n for f, n in ((TL, "two_level"), (OP, "one_pass"), (NS, "no_skip")) if flags & f) or "default"


def _nonempty_parts(n, vparts, vramp):
    cut = H.part_boundaries(n, vparts, vramp / 100)
    return sum(1 for q in range(vparts) if cut[q + 1] > cut[q])


# ---- 1. every pattern through every pass shape ------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", P.PATTERNS)
def test_pattern_sorts_bit_exact(name, n):
    a, want = _case(name, n)
    for flags in SHAPES:
        got, st = _sort(a, flags)
        _assert_same(got, want, name, n, flags)
        assert st.skipped == _expected_skips(a["key"], flags), (name, n, flags)


RADIX_PATTERNS = ["descending", "heavy_0.9", "all_but_one_mid", "all_but_one_last", "bit63_only", "runs_2817", "saw_2816",
                  "few_257", "supertile_segments"]


@pytest.mark.parametrize("radix", [8, 11, 13])
@pytest.mark.parametrize("name", RADIX_PATTERNS)
def test_pattern_radix_widths(name, radix):
    # radix 8: one partition step per pass; 11: 5 + 6 bit steps or one-pass with a 3-bit high part; 13: a 12-bit last digit
    n = P.SUPERTILE + 1
    a, want = _case(name, n)
    for flags in (0, TL, OP, TL | OP):
        got, st = _sort(a, flags, radix)
        _assert_same(got, want, name, radix, flags)
        assert st.skipped == _expected_skips(a["key"], flags, radix), (name, radix, flags)


PAYLOAD_PATTERNS = ["heavy_0.9", "all_but_one_mid", "bit0_only", "runs_32", "runs_2817", "runs_5633", "saw_2816", "few_2",
                    "few_257", "supertile_segments", "lying_sample"]


@pytest.mark.parametrize("vals", ["small", "zero"])
@pytest.mark.parametrize("name", PAYLOAD_PATTERNS)
def test_pattern_repeated_payloads(name, vals):
    # vals in [0, 16) or all zero: equal (key, val) records, so verify() (strictly increasing) does not apply; the
    # multiset and the stable sort by key still pin the output
    n = P.SUPERTILE + 1
    a, want = _case(name, n, vals)
    for flags in (0, TL, OP, TL | OP):
        with lsb.DistributedSorter(n, flags=flags) as s:
            s.upload(a)
            assert s.checksum() == O.checksum(a)
            s.my_sort()
            assert s.checksum() == O.checksum(a), (name, vals, flags)
            _assert_same(s.download(), want, name, vals, flags)


# ---- 2. pass by pass ----------------------------------------------------------------------------------------------------
PASS_PATTERNS = ["ascending", "heavy_0.999", "all_but_one_first", "all_but_one_last", "bit0_only", "runs_5633", "saw_65536",
                 "few_2", "supertile_segments", "lying_sample"]


@pytest.mark.parametrize("flags", [0, TL, OP, TL | OP], ids=_shape)
@pytest.mark.parametrize("name", PASS_PATTERNS)
def test_pattern_each_pass(name, flags):
    """counts, starts and the array after every lsb_pass against the oracle's single pass; steps and skips per pass"""
    n = P.SUPERTILE + 1
    cur, _ = _case(name, n)
    parts = _nonempty_parts(n, 16, 130) if flags & TL else 1
    with lsb.DistributedSorter(n, flags=flags) as s:
        s.upload(cur)
        for p in range(4):
            want, counts, starts, _ = O.one_pass(cur, n, 1, 16, p)
            assert (s.histogram(p) == counts[0]).all(), (name, flags, p)
            assert (s.starts(p) == starts[:, 0]).all(), (name, flags, p)
            st = s.global_shuffle(p)
            skips = _expected_skips(cur["key"], flags, passes=[p])
            steps = 1 if flags & OP else 2
            assert st.passes == 1 and st.skipped == skips, (name, flags, p)
            assert st.subpasses == parts * (steps - skips if not flags & TL else steps * (1 - skips)), (name, flags, p)
            cur = s.download()
            _assert_same(cur, want, name, flags, p)


# ---- 3. the 16-bit shared-memory counters of digit_hist_kernel past their spill point -----------------------------------
# digit_hist_kernel counts in packed 16-bit shared counters; one that reaches 0x8000 moves 0x8000 to the global table
# (dh_add, csrc/lsb_onepass.cuh).  A CTA of a one-digit count (lsb_histogram, lsb_starts, count_parts) reads the 8192-
# element chunks c, c + groups, ... with groups = min(SMs / 1 role, chunks) (launch_digit_hist, csrc/lsbsort.cu).
# At n = 3 * 2^22 + 13 on a B200 (148 SMs) there are 1536 full chunks, so every CTA reads >= 10 of them = 81 920
# elements and a heavy key at f >= 0.9 puts >= 73 700 of them in one bin: each such counter spills twice, and a
# counter without the spill would wrap at 65 536.  (At 2^23 + 13 a CTA reads <= 57 344 elements: the guard trips,
# but 16 bits would hold the count.)  _assert_counters_wrap_without_spill repeats this with the device's SM count.
# The one-pass shape counts its 4 digits in 4 roles of 37 CTAs, >= 41 chunks each: about nine spills per counter.
SPILL_N = 3 * (1 << 22) + 13
SPILL_PATTERNS = ["heavy_0.9", "heavy_0.999", "all_but_one_mid"]


def _assert_counters_wrap_without_spill(m, f=0.9):
    """the least a CTA of a one-digit count over m elements puts into the heavy bin must pass 65 536"""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    full_chunks = m // 8192
    groups = max(1, min(sms, -(-m // 8192)))
    least = f * (full_chunks // groups) * 8192
    assert least > 65536 + 1000, f"{sms} SMs: a CTA counts only {least:.0f} of the heavy bin; make SPILL_N larger"


@pytest.mark.parametrize("name", SPILL_PATTERNS)
def test_spill_counts(name, lib_tune):
    """histogram() and starts() only -- the counts are checked before anything is scattered by them"""
    _assert_counters_wrap_without_spill(SPILL_N)
    a = P.make(name, SPILL_N)
    keys = a["key"]
    for radix in (16, 11):
        with lsb.DistributedSorter(SPILL_N, radix_bits=radix) as s:
            s.upload(a)
            for p in range(s.num_passes()):
                bits = s.digit_bits(p)
                want = np.bincount(P.digit(keys, radix * p, bits), minlength=1 << bits)
                assert want.max() > 0.89 * SPILL_N
                assert (s.histogram(p) == want).all(), (name, radix, p)
                assert (s.starts(p) == np.cumsum(want) - want).all(), (name, radix, p)
    # the virtual-rank pass counts each part into u32 bins (count_parts).  One part is the whole shard, as above: a
    # counter without the spill would wrap.  Two parts of 6.3 M give a CTA <= 49 152 elements: the guard trips, but
    # only vparts = 1 would catch a missing spill.  16 parts would not trip the guard at all.
    for vparts in (1, 2):
        lib_tune("vparts", vparts)
        with lsb.DistributedSorter(SPILL_N, flags=TL) as s:
            s.upload(a)
            for p in range(4):
                want = np.bincount(P.digit(keys, 16 * p, 16), minlength=65536)
                assert (s.starts(p) == np.cumsum(want) - want).all(), (name, vparts, p)


@pytest.mark.parametrize("name", SPILL_PATTERNS)
def test_spill_sorts_and_skips(name):
    a = P.make(name, SPILL_N)
    want = P.reference(a)
    for flags in SHAPES:
        got, st = _sort(a, flags)
        _assert_same(got, want, name, flags)
        # a digit that is constant over all 12.6 M elements is skipped; the digit of the one odd element is not
        skips = _expected_skips(a["key"], flags)
        if name.startswith("all_but_one"):
            assert skips == (0 if flags & NS else 3 if flags & (TL | OP) else 7)
        else:
            assert skips == 0
        assert st.skipped == skips, (name, flags)


# ---- 4. the virtual-rank pass (FLAG_TWO_LEVEL): part cuts and exchange tunables ----------------------------------------
# (16, 300) at 65 536 leaves part 0 empty and several parts of 32 elements; (16, 298) at 65 546 empties part 14 between
# two sorted parts; 65 535 is below the ramp threshold (V * 4096) and cuts equal parts
VR_CUTS = [(1, 130), (2, 130), (3, 100), (5, 300), (16, 100), (16, 101), (16, 300), (16, 298)]
VR_SIZES = [65535, 65536, 65546, (1 << 20) + 77]


@pytest.mark.parametrize("flags", [TL, TL | OP], ids=_shape)
@pytest.mark.parametrize("data", ["random", "heavy_0.9", "lying_sample"])
@pytest.mark.parametrize("vparts,vramp", VR_CUTS)
def test_virtual_rank_part_cuts(vparts, vramp, data, flags, lib_tune):
    lib_tune("vparts", vparts)
    lib_tune("vramp", vramp)
    for n in VR_SIZES:
        a, want = _case(data, n)
        got, st = _sort(a, flags)
        _assert_same(got, want, vparts, vramp, data, flags, n)
        # every non-empty part is sorted once per pass (two steps, or one one-pass launch), no empty part is
        assert st.skipped == 0 and st.subpasses == 4 * _nonempty_parts(n, vparts, vramp) * (1 if flags & OP else 2), \
            (vparts, vramp, data, flags, n, st.subpasses)


@pytest.mark.parametrize("radix,flags", [(8, TL), (11, TL | OP)], ids=["radix8", "radix11-one_pass"])
def test_virtual_rank_empty_interior_part(radix, flags, lib_tune):
    # a part sorted in one launch (a digit of <= 8 bits, or the one-pass shape) goes to one of two scratches until its
    # exchange has read it; part 14 is empty, so parts 13 and 15 are sorted one after the other and must not share one
    lib_tune("vparts", 16)
    lib_tune("vramp", 298)
    n = 65546
    parts = _nonempty_parts(n, 16, 298)
    assert parts == 14
    for data in ("random", "heavy_0.9", "lying_sample"):
        a, want = _case(data, n)
        got, st = _sort(a, flags, radix)
        _assert_same(got, want, radix, data, flags)
        assert st.subpasses == H.num_passes(radix) * parts, (radix, data, st.subpasses)


TUNABLE_RUNS = [("ex_threads", 256, TL), ("ex_u", 8, TL), ("ex_ctas", 3, TL), ("ex_ctas", 3, TL | OP), ("op_ctas_mgpu", 1, TL | OP),
                ("op_ctas_mgpu", 4, TL | OP), ("op_hints", 0, OP), ("op_hints", 0, TL | OP)]


@pytest.mark.parametrize("key,value,flags", TUNABLE_RUNS, ids=[f"{k}={v}-{_shape(f)}" for k, v, f in TUNABLE_RUNS])
def test_exchange_and_onepass_tunables(key, value, flags, lib_tune):
    lib_tune(key, value)
    n = (1 << 20) + 77
    for data in ("heavy_0.9", "lying_sample"):
        a, want = _case(data, n)
        got, st = _sort(a, flags)
        _assert_same(got, want, key, value, flags, data)
        assert st.subpasses == (4 * _nonempty_parts(n, 16, 130) * (1 if flags & OP else 2) if flags & TL else 4)


# ---- 5. the fused next-digit count on skewed data ------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [TL, TL | OP], ids=_shape)
def test_fusion_follows_the_sample(flags):
    """lying_sample: plan_fusion sees a wide digit 1 in the first 65 536 elements, so pass 0's exchange counts digit 1
    -- and then every element after the sample lands in one bin (the exchange's warp-uniform slot and held-run paths).
    The same multiset reversed shows the one-bin part first: no fusion for pass 1, which then counts its own digit
    (one more count launch per part)."""
    n = (1 << 20) + 77
    a, want = _case("lying_sample", n)
    got, st = _sort(a, flags)
    _assert_same(got, want, "lying", flags)
    skewed = a[::-1].copy()
    got2, st2 = _sort(skewed, flags)
    _assert_same(got2, P.reference(skewed), "skewed", flags)
    assert st.kernel_launches < st2.kernel_launches, (st.kernel_launches, st2.kernel_launches)
