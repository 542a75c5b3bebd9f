"""The decisive inputs of tests/decisive.py without a GPU: the decoders invert the key orders, the fault-free model of
every plan the GPU module runs equals an independent reference, every fault of every step at every radix and in every
shape changes the output of the block the GPU inputs contain, and on data where the final output hides early steps the
checker says so."""
import numpy as np
import pytest

import decisive as D
import key_orders as KO
import lexsort_ref as R
import narrow_keys as NK
import patterns as P


# ---- decoders ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", R.NAMES)
def test_decode_inverts_the_order(name):
    w = R.WIDTH[name]
    rng = np.random.default_rng(w)
    raw = R.special_mix(4096, name, seed=1)
    for desc in (False, True):
        keys = D.encode(raw, name, desc)
        back = D.decode(keys, name, desc)
        assert np.array_equal(D.encode(back, name, desc), keys), desc  # same key, so the same place in every sort
        x = R.typed(raw, name)
        plain = x == x if np.issubdtype(x.dtype, np.integer) else ~np.isnan(x) & (x != 0)
        assert np.array_equal(back[plain], raw[plain]), desc  # every pattern but NaNs and zeros comes back as it was
        words = rng.integers(0, 1 << w, 4096, dtype=np.uint64) if w < 64 else rng.integers(0, 1 << 64, 4096, dtype=np.uint64)
        once = D.encode(D.decode(words, name, desc), name, desc)
        assert np.array_equal(D.encode(D.decode(once, name, desc), name, desc), once)
        assert (once == words).mean() > 0.96, desc  # only the NaN ranges (3 % of float16's words) and -0.0 move


# ---- the plans the GPU module runs, each on the block its inputs contain ---------------------------------------------------
def _plans():
    out = {f"sort-{o}": (D.sort_plan(*nd), range(1, 17)) for o, nd in D.WIDE_ORDERS.items()}
    out.update({f"sort-{x}-{'desc' if d else 'asc'}": (D.sort_plan(x, d), range(1, 17)) for x in NK.NAMES for d in (False, True)})
    out.update({f"lexsort-{'-'.join(names)}": (D.lexsort_plan(names, d), range(1, 17)) for names, d in D.LEXSORTS})
    out.update({f"segments-{x}-r{r}": (D.segment_plan(x, d, D.segment_bits(r)), [r]) for x, d in D.SEGMENT_KEYS
                for r in range(1, 17)})
    return out


PLANS = _plans()


def _reference(plan):
    g = plan.given
    if "cols" in g:
        return R.reference(g["cols"], g["names"], g["descending"])
    if "seg" in g:
        return np.lexsort((R.ranks(g["raw"], g["name"], g["descending"]), g["seg"]))
    if R.WIDTH[g["name"]] == 64:
        return KO.argsort(g["raw"], KO.ORDERS[next(o for o, nd in D.WIDE_ORDERS.items() if nd == (g["name"], g["descending"]))])
    return NK.argsort(g["raw"], g["name"], g["descending"])


@pytest.mark.parametrize("what", sorted(PLANS))
def test_model_equals_reference(what):
    """the rounds' key words sort like the independent reference, the steps of every radix and shape tile each round,
    and step by step the model sorts the same (at a radix of at most 8 bits and at one above)"""
    plan, radices = PLANS[what]
    want = _reference(plan)
    assert np.array_equal(plan.order(), want)
    for radix in radices:
        for shape in D.SHAPES:
            for k, rd in enumerate(plan.rounds):
                spans = [(s, w) for j, s, w, _ in D.steps(plan, radix, shape) if j == k]
                assert spans[0][0] == 0 and all(a + w == b for (a, w), (b, _) in zip(spans, spans[1:]))
                assert spans[-1][0] + spans[-1][1] >= rd.live and spans[-1][0] < rd.live
    picks = radices if len(radices) == 1 else [3 + len(what) % 6, 9 + len(what) % 8]
    for radix in picks:
        for shape in D.SHAPES:
            assert np.array_equal(D.lsd(plan, radix, shape), want), (radix, shape)


@pytest.mark.parametrize("what", sorted(PLANS))
def test_every_fault_changes_the_output(what):
    plan, radices = PLANS[what]
    assert D.Checker(plan).undetected(radices) == []


def test_fast_check_equals_the_faulty_sort():
    """the composite-key check and the faulty output from three sorts agree with the faulted sort run step by step"""
    rng = np.random.default_rng(7)
    plans = [D.sort_plan("float64", False, n=3000), D.sort_plan("float32", True, n=3000),
             D.lexsort_plan(("float64", "int16"), (True, False), n=3000), D.segment_plan("int32", True, 5, n=3000)]
    raw = rng.integers(0, 1 << 64, 3000, dtype=np.uint64)  # uniform keys: many faults leave the output alone
    plans.append(D.Plan([D.key_round(raw, "int64", False)], raw=raw, name="int64", descending=False))
    seen = {True: 0, False: 0}
    for plan in plans:
        c = D.Checker(plan)
        for _ in range(60):
            radix, shape = int(rng.integers(1, 17)), D.SHAPES[int(rng.integers(0, 3))]
            st = D.steps(plan, radix, shape)
            i = int(rng.integers(0, len(st)))
            for f in D.faults(plan, st[i]):
                got = D.lsd(plan, radix, shape, f, i)
                assert np.array_equal(c.faulty_output(st[i], f), got), (radix, shape, st[i], f)
                assert c.detected(st[i], f) == (not np.array_equal(got, c.correct)), (radix, shape, st[i], f)
                seen[c.detected(st[i], f)] += 1
    assert seen[True] > 100 and seen[False] > 100


def test_gpu_inputs_hold_the_block():
    for radix in (1, 4, 5, 16):
        n = D.gpu_count(radix)
        assert n > P.SUPERTILE + D.BLOCK or radix <= 4
        big, blk = D.sort_plan("float64", True, n), D.sort_plan("float64", True)
        starts = D.block_starts(n)
        assert starts[-1] == n - D.BLOCK and starts[0] < (P.SUPERTILE if radix > 4 else 6 * P.PART_TILE) < starts[0] + D.BLOCK
        for s in starts:
            assert np.array_equal(big.given["raw"][s:s + D.BLOCK], blk.given["raw"])
        names, desc = D.LEXSORTS[-1]
        big, blk = D.lexsort_plan(names, desc, n), D.lexsort_plan(names, desc)
        for a, b in zip(big.given["cols"], blk.given["cols"]):
            assert np.array_equal(a[starts[0]:starts[0] + D.BLOCK], b)
        big, blk = D.segment_plan("float32", False, D.segment_bits(radix), n), D.segment_plan("float32", False, D.segment_bits(radix))
        for s in starts:  # the block's records keep their relative order among the others
            keep = (big.given["src"] >= s) & (big.given["src"] < s + D.BLOCK)
            assert np.array_equal(big.given["raw"][keep], blk.given["raw"])
            assert np.array_equal(big.given["seg"][keep], blk.given["seg"])


# ---- the checker finds blind steps --------------------------------------------------------------------------------------------
def _blind(plan, radix, shape="two_step"):
    return sorted({i for _, _, i, _, _ in D.Checker(plan).undetected([radix], [shape])})


def test_uniform_keys_hide_the_first_steps():
    """uniform random uint64: no two of 2^15 keys agree on the top 48 bits, so nothing the low steps do shows"""
    raw = np.random.default_rng(1).integers(0, 1 << 64, D.BLOCK, dtype=np.uint64)
    plan = D.Plan([D.key_round(raw, "uint64", False)])
    blind = _blind(plan, 16)
    assert blind[0] == 0 and 0 < len(blind) < len(D.steps(plan, 16, "two_step")) - 2
    assert _blind(D.sort_plan("uint64", False), 16) == []


def test_few_valued_lexsort_columns_hide_round_0():
    """the columns of test_gpu_lexsort.test_pass_shapes_and_radices' (int32, float32, uint16) mix: five values in each
    of the first two columns, so pairs equal above a step of their round and different in it do not exist"""
    names = ("int32", "float32", "uint16")
    cols = [R.few_values(D.BLOCK, x, k=5, seed=c) if c < len(names) - 1 else R.special_mix(D.BLOCK, x, seed=c)
            for c, x in enumerate(names)]
    plan = D.lexsort_columns(cols, names, (False, True, False))
    st = D.steps(plan, 13, "two_step")
    round0 = [i for i, s in enumerate(st) if s[0] == 0]
    assert len(round0) == 10 and set(round0) <= set(_blind(plan, 13))
    assert _blind(D.lexsort_plan(names, (False, True, False)), 13) == []
    assert np.array_equal(plan.order(), R.reference(cols, names, (False, True, False)))
