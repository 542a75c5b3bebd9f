"""The decisive inputs of tests/unique_decisive.py without a GPU: the mixes reach every kernel instance, the fault-free
model equals the independent reference, every fault of the model changes the output of every input the GPU module runs
(both modes, both directions), the inputs hold single-bit neighbours, twins and group starts where the module says, and
on the data of test_gpu_unique.test_pass_shapes_and_radices the checker finds the blind bits."""
import numpy as np
import pytest

import lexsort_ref as R
import patterns as P
import unique_decisive as U
import unique_ref as UR
from test_gpu_lexsort import ROUND_MIXES

CASES = sorted(U.cases())


def _model(mix, flipped, consecutive):
    names, desc = U.cases()[mix, flipped]
    b, cols = U.block_input(mix, flipped, consecutive)
    return b, cols, U.Model(cols, names, desc, consecutive)


def test_mixes_reach_every_kernel_instance():
    """every type in both directions in an earlier round and in the last round; 1, 2 and 3 rounds; rounds of 1-4
    columns in the flag kernel and in the tile kernel"""
    earlier, last, nrounds, flag_cols, tile_cols = set(), set(), set(), set(), set()
    for names, desc in U.cases().values():
        rs = U.rounds(names)
        nrounds.add(len(rs))
        for r, (first, ncols, _, _) in enumerate(rs):
            (last if r == len(rs) - 1 else earlier).update(zip(names[first:first + ncols], desc[first:first + ncols]))
            (tile_cols if r == len(rs) - 1 else flag_cols).add(ncols)
    every = {(x, d) for x in R.NAMES for d in (False, True)}
    assert earlier == every and last == every
    assert nrounds == {1, 2, 3} and flag_cols == {1, 2, 3, 4} and tile_cols == {1, 2, 3, 4}


@pytest.mark.parametrize("mix,flipped", CASES)
def test_model_equals_reference(mix, flipped):
    names, desc = U.cases()[mix, flipped]
    for consecutive in (False, True):
        _, cols, m = _model(mix, flipped, consecutive)
        assert m.n == U.BLOCK_N
        u, index, inverse, counts = m.result()
        want = UR.reference(cols, names, list(desc), consecutive)
        assert u == len(want[0])
        assert np.array_equal(index, want[0]) and np.array_equal(inverse, want[1]) and np.array_equal(counts, want[2])
        assert (m.correct[1][u:] == U.SENTINEL).all() and (m.correct[3][u:] == U.SENTINEL).all()


@pytest.mark.parametrize("mix,flipped", CASES)
def test_every_fault_changes_the_output(mix, flipped):
    for consecutive in (False, True):
        b, _, m = _model(mix, flipped, consecutive)
        fs = U.faults(m, b.lost)
        assert len(fs) > 30
        assert U.Checker(m).undetected(fs) == [], (mix, flipped, consecutive)


@pytest.mark.parametrize("mix,flipped", CASES)
def test_unreachable_bits(mix, flipped):
    """sorted mode misses exactly the top bit of every float column with no float column above it (its single-bit
    neighbours would span 2^W - 1 words, more than a float has); consecutive mode misses nothing"""
    names, desc = U.cases()[mix, flipped]
    want = [(c, R.WIDTH[x] - 1) for c, x in enumerate(names) if x in U.FLOATS and not any(y in U.FLOATS for y in names[c + 1:])]
    assert U.Block(names, desc, False).lost == want
    assert U.Block(names, desc, True).lost == []


@pytest.mark.parametrize("mix,flipped", CASES)
def test_inputs_hold_neighbours_twins_and_starts(mix, flipped):
    names, desc = U.cases()[mix, flipped]
    sh = U.shifts(names)
    last = len(U.rounds(names)) - 1
    for consecutive in (False, True):
        b, cols, m = _model(mix, flipped, consecutive)
        lost = {(sh[c][0], sh[c][1] + bit) for c, bit in b.lost}
        every = {(r, bit) for r, (_, _, bits, _) in enumerate(m.rounds) for bit in range(bits)}
        assert set(U.Checker(m).mask_undetected()) == lost  # single-bit neighbours at every other bit of every round
        h, p = m.correct_heads, m.pos
        assert len(lost) <= 1 and every - lost
        for res in range(U.WARP):  # starts and non-starts on every lane
            assert h[p % U.WARP == res].any() and not h[p % U.WARP == res].all()
        for t in range(1, -(-m.n // U.TILE)):  # tile starts and their neighbours, both ways
            assert h[t * U.TILE - 1:t * U.TILE + 2].all() if t % 2 else not h[t * U.TILE - 1:t * U.TILE + 2].any()
        assert all(h[t * U.TILE:(t + 1) * U.TILE].any() for t in range(-(-m.n // U.TILE)))
        x = [np.concatenate([[np.uint64(0)], w[1:] ^ w[:-1]]) for w in m.W]
        for r in range(last + 1):  # a start of round r alone on lane 0, and one on lane 31 with a run after it
            only = h & np.all([(x[q] != 0) == (q == r) for q in range(last + 1)], axis=0)
            assert (only & (p % U.WARP == 0)).any()
            at31 = np.flatnonzero(only & (p % U.WARP == 31))
            assert (at31 + 1 < m.n).any() and not h[at31[at31 + 1 < m.n] + 1].all()
        for c, x_ in enumerate(names):  # twins: equal keys with other bits next to each other, at +0.0 and at NaN
            if x_ not in U.FLOATS:
                continue
            raw = cols[c][m.order]
            sp = U.special_raws(x_)
            same = ~h[1:] & (raw[1:] != raw[:-1])
            assert (same & (raw[1:] == sp["negzero"]) | same & (raw[:-1] == sp["negzero"])).any(), (x_, consecutive)
            assert (same & np.isin(raw[1:], sp["nans"])).any(), (x_, consecutive)


def test_head_faults_checked_on_flags_equal_whole_outputs():
    b, _, m = _model(8, True, False)
    c = U.Checker(m)
    fs = U.faults(m, b.lost) + [("mask", r, bit) for r, bit in [(1, 63), (0, 0)]]
    assert all(c.detected(f) == c.detected_full(f) for f in fs)
    m2 = U.Model([R.few_values(5000, "int32", 3, seed=1)], ["int32"], [False], False)
    c2 = U.Checker(m2)
    for f in U.faults(m2):
        assert c2.detected(f) == c2.detected_full(f), f
    assert sorted(c2.mask_undetected()) == sorted(f[1:] for f in U.faults(m2) if f[0] == "mask" and not c2.detected(f))


@pytest.mark.parametrize("mix", [2, 6])
def test_large_inputs_place_the_grid_stride_boundaries(mix):
    """for every SM count from 16 to 170: a start of each earlier round alone on a grid-stride boundary and on an IO_U
    step boundary, a non-start on each; on the 148-SM B200 every grid fault of the model changes the output"""
    for consecutive in (False, True):
        names, desc = U.cases()[mix, False]
        b = U.Block(names, desc, consecutive)
        kinds = b.kinds()
        for sms in range(16, 171):
            stride = U.grid_stride(sms, U.LARGE_N)
            assert stride == sms * U.IO_CTAS_PER_SM * U.IO_THREADS and 12 * stride < U.LARGE_N
            starts = np.concatenate([[0], np.cumsum(U.large_lengths(b, stride))[:-1]])
            at = {int(s): g for g, s in enumerate(starts)}
            targets = U.grid_targets(b, stride, U.LARGE_N)
            assert {r for r in targets.values() if r is not None} == set(range(len(U.rounds(names)) - 1))
            for p, r in targets.items():
                assert (p in at) == (r is not None) and (r is None or kinds[at[p]] == {r}), (sms, p, r)
        b, cols, stride = U.large_input(mix, False, consecutive, 148)
        m = U.Model(cols, names, desc, consecutive, stride)
        grid = [f for f in U.faults(m, b.lost) if f[0] == "grid"]
        assert len(grid) == 8 and U.Checker(m).undetected(grid) == []


@pytest.mark.parametrize("mix", [0, 2, 7])
def test_few_values_hide_most_bits(mix):
    """the data of test_gpu_unique.test_pass_shapes_and_radices (four values per column, sorted mode): neighbouring
    groups differ in many bits at once, so a head test that ignored one bit would pass there for most bits of every
    round; the decisive blocks leave none out"""
    names = ROUND_MIXES[mix]
    n = P.SUPERTILE + 1
    cols = [R.few_values(n, x, k=4, seed=c) for c, x in enumerate(names)]
    m = U.Model(cols, names, [c % 2 == 1 for c in range(len(names))], False)
    blind = U.Checker(m).mask_undetected()
    for r, (_, _, bits, _) in enumerate(m.rounds):
        assert sum(1 for q, _ in blind if q == r) >= bits - 1, (r, bits)  # 63 of 64, 16 of 16, or all
