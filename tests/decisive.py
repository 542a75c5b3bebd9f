"""Inputs on which every step of the LSD sort is decisive, and the fault model that proves it.

An LSD sort hides its early steps behind its late ones: two records that differ in a high digit end up in the right order
whatever the earlier steps did with them.  A comparison of the final output sees a faulty step only if the input has
records that are equal above that step and differ in it.  The inputs here have such pairs at every bit.

Words.  Records are drawn as words of `width` bits in order-key space (the key word the passes sort, or several of
them side by side).  Each record takes one of `BASES` random bases, keeps its bits at and above a cut c, and draws its
bits below c at random; c is uniform over 1..width, and a few records have c = 0 (exact copies: stability).  Records
of one base whose cut is b + 1 are equal above bit b and differ at it (half the time), whatever the radix or the step.

Decoders turn the words into raw bit patterns of the ten key types, in both directions (the inverses of order_key and
order_narrow).  A pattern that does not encode back to its word (NaNs with other payloads or signs, -0.0) is replaced by
the one that encodes to the same key (one NaN, +0.0): those records become ties, which harms nothing.  A lexsort's columns are slices of one wide word, the most
significant column on top; a segmented sort's segment id is the word's top field, and the records are stably sorted by
it to give the offsets.

Plans and steps.  A plan is the list of rounds of stable passes a call makes (one for a sort, one per lexsort round,
key passes then segment passes for segments), each on its own key word.  `steps` lists a round's steps at a radix in
one of three shapes: "two_step" (a digit over 8 bits as two balanced sub-steps), "one_pass" (its low byte, then the
rest) and "digit" (the whole digit: the two-level shape's exchange), all from hostlogic.plan_pass.

Faults.  One step of one plan is faulted: it is skipped, it reads its digit one bit too high or too low, it merges
bins 2k and 2k + 1, it reverses the order of the records it ties, a narrow key's clamped last digit is read unclamped
(into the raw key the word holds from bit 32), or an ordered key's step reads the raw bits instead of the order key.
Each is a pairwise fault: whether the faulty sort puts one record before another depends only on their two key words
and their input order.  So a pair that a fault misorders in a block misorders it in any larger input that holds the
block's records in the same relative order, as a contiguous run or spread between other records.  That lets a CPU
prove a block of BLOCK records and the GPU sort larger inputs built around copies of it.

The faulty output is a stable sort by the bits below the step, then the faulted step, then a stable sort by the bits
above it.  Written as one composite key (rank above, faulted digit, rank below), it equals the correct output exactly
when that key increases along the correct order: one pass over the records, no sort per fault.
"""
import zlib

import numpy as np

import lexsort_ref as R
import narrow_keys as NK
import patterns as P
from distributed_lsb_b200 import hostlogic as H
from test_lexsort_cpu import order

BLOCK = 1 << 15          # records the CPU proves
BASES = 32
COPIES = 0.03            # share of records with cut 0
SHAPES = ("two_step", "one_pass", "digit")
ALL = (1 << 64) - 1

# what the GPU module sorts: 64-bit keys through the context's order (records, pass by pass, segments), the narrow
# types with the direction alternating by radix, lexsort rounds of 16, 32, 48 and 64 bits and one of 64 | 64 | 48, and
# segments (2^(radix + 1) of them: two segment passes at every radix) of a 64-bit and a narrow key
WIDE_ORDERS = {"u64": ("uint64", False), "i64_desc": ("int64", True), "f64": ("float64", False),
               "f64_desc": ("float64", True)}
LEXSORTS = [(("bfloat16",), (True,)),
            (("int16", "float16"), (False, True)),
            (("float32", "uint16"), (True, False)),
            (("uint16", "int16", "bfloat16", "float16"), (False, True, True, False)),
            (("float64", "int64", "int32", "float16"), (True, False, True, False))]
SEGMENT_KEYS = [("float64", True), ("float32", False)]


def narrow_descending(name, radix):
    return (radix + NK.NAMES.index(name)) % 2 == 1


def segment_bits(radix):
    return radix + 1


def gpu_count(radix):
    """records of a GPU input: the one-pass shape runs two supertiles and more; 16-64 passes (radix <= 4) sort fewer"""
    return 3 * BLOCK + 77 if radix <= 4 else P.SUPERTILE + 2 * BLOCK + 7


def _mask(w):
    return np.uint64((1 << w) - 1 if w < 64 else ALL)


# ---- words ---------------------------------------------------------------------------------------------------------------
def prefix_family(n, width, seed):
    """n words of `width` bits as limbs (uint64 arrays, least significant first): one of BASES bases above a cut drawn
    from 1..width (0 for a share COPIES), random bits below it"""
    rng = np.random.default_rng([seed, n, width])
    nl = -(-width // 64)
    base = rng.integers(0, 1 << 64, (nl, BASES), dtype=np.uint64)
    b = rng.integers(0, BASES, n)
    cut = rng.integers(1, width + 1, n)
    cut[rng.random(n) < COPIES] = 0
    limbs = []
    for j in range(nl):
        k = np.clip(cut - 64 * j, 0, 64).astype(np.uint64)
        low = np.where(k == 64, np.uint64(ALL), (np.uint64(1) << np.minimum(k, 63)) - np.uint64(1))
        top = width - 64 * j
        word = (base[j][b] & ~low) | (rng.integers(0, 1 << 64, n, dtype=np.uint64) & low)
        limbs.append(word & _mask(min(top, 64)))
    return limbs


def field(limbs, lo, w):
    """bits [lo, lo + w) of limb words, w <= 64"""
    j, s = divmod(lo, 64)
    v = limbs[j] >> np.uint64(s)
    if s and s + w > 64 and j + 1 < len(limbs):
        v = v | (limbs[j + 1] << np.uint64(64 - s))
    return v & _mask(w)


def block_starts(n):
    """where copies of the proven block sit in an input of n records: across a tile boundary (the one-pass supertile's
    when there is room, a partition tile's otherwise) and at the end"""
    if n == BLOCK:
        return [0]
    edge = P.SUPERTILE if n >= P.SUPERTILE + 2 * BLOCK else P.PART_TILE * (BLOCK // P.PART_TILE + 1)
    starts = [edge - BLOCK // 2, n - BLOCK]
    assert starts[0] + BLOCK <= starts[1], n
    return starts


def words(n, width, seed):
    """the proven block (n == BLOCK; a smaller family below), or n records of another prefix family with copies of the
    block at block_starts"""
    if n <= BLOCK:
        return prefix_family(n, width, seed)
    blk = prefix_family(BLOCK, width, seed)
    out = prefix_family(n, width, seed + 1)
    for s in block_starts(n):
        for o, b in zip(out, blk):
            o[s:s + BLOCK] = b
    return out


# ---- decoders --------------------------------------------------------------------------------------------------------------
def decode(w, name, descending):
    """order keys (the low width bits of `w`) -> raw bit patterns of the type whose order key they are; where no pattern
    encodes to a word (the NaN ranges but one word, the word of -0.0) the pattern of the word it does encode to (one NaN,
    +0.0)"""
    raw = _decode(w, name, descending)
    return _decode(encode(raw, name, descending), name, descending)


def _decode(w, name, descending):
    width = R.WIDTH[name]
    allb, sign = _mask(width), np.uint64(1 << (width - 1))
    k = np.asarray(w, dtype=np.uint64) & allb
    if descending:
        k = ~k & allb
    if name.startswith("int"):
        k = k ^ sign
    elif name.startswith("float") or name == "bfloat16":
        k = np.where(k & sign, k ^ sign, ~k & allb)
    return k.astype(R.UINT[width])


def encode(raw, name, descending):
    return order(raw, name, descending).astype(np.uint64)


# ---- plans -----------------------------------------------------------------------------------------------------------------
class Round:
    """one run of stable passes: `word` is the key word the passes read (order key in the low `bits` bits; a narrow
    key's raw bits from bit `above` on), `live` the bits that can differ (a segment id's; the passes cover them rounded up
    to whole digits), `raw` what a step reads if it skips the key order"""

    def __init__(self, word, bits, live=None, above=None, raw=None, pad=False):
        self.word, self.bits, self.above, self.raw, self.pad = word, bits, above, raw, pad
        self.live = bits if live is None else live
        self.key = word & _mask(bits)

    def plan_bits(self, radix):
        return -(-self.live // radix) * radix if self.pad else self.bits


def key_round(raw, name, descending):
    """the passes of a sort of `raw` keys: the context's 64-bit plan (reading order_key of the raw key) or a narrow
    key's W-bit plan (the pack's word: raw key at bit 32, order key below)"""
    width = R.WIDTH[name]
    ok = encode(raw, name, descending)
    if width == 64:
        return Round(ok, 64, raw=raw.astype(np.uint64))
    return Round(raw.astype(np.uint64) << np.uint64(32) | ok, width, above=32)


class Plan:
    """rounds (least significant first) over n records, and what the GPU call is given"""

    def __init__(self, rounds, **given):
        self.rounds = rounds
        self.n = len(rounds[0].word)
        self.given = given

    def order(self):
        """the correct output: the stable sort by the rounds' key words"""
        return np.lexsort([r.key for r in self.rounds])


def _seed(*what):
    return zlib.crc32(repr(what).encode())


def sort_plan(name, descending, n=BLOCK):
    """lsb_sort_device / lsb_sort (64-bit keys through the context's order) or lsb_sort_device_typed (narrow keys)"""
    raw = decode(words(n, R.WIDTH[name], _seed("sort", name, descending))[0], name, descending)
    return Plan([key_round(raw, name, descending)], raw=raw, name=name, descending=descending)


def lexsort_columns(cols, names, descending):
    """the plan of lsb_lexsort_device on bit-pattern columns (columns[0] least significant)"""
    widths = [R.WIDTH[x] for x in names]
    rounds = []
    for first, ncols, bits, _ in H.lexsort_rounds(widths, 16):
        w, at = np.zeros(len(cols[0]), dtype=np.uint64), 0
        for c in range(first, first + ncols):
            w |= encode(cols[c], names[c], descending[c]) << np.uint64(at)
            at += widths[c]
        rounds.append(Round(w, bits))
    return Plan(rounds, cols=cols, names=tuple(names), descending=tuple(descending))


def lexsort_plan(names, descending, n=BLOCK):
    """column c is the slice of one wide word above the columns below it"""
    widths = [R.WIDTH[x] for x in names]
    limbs = words(n, sum(widths), _seed("lexsort", names, descending))
    at = np.cumsum([0] + widths)
    cols = [decode(field(limbs, int(at[c]), widths[c]), x, d) for c, (x, d) in enumerate(zip(names, descending))]
    return lexsort_columns(cols, names, descending)


def segment_plan(name, descending, segbits, n=BLOCK):
    """lsb_sort_segments_device(_typed) over 2^segbits segments: (segment, key) drawn as one word, the records stably
    sorted by segment (a block inside a larger input keeps its records' relative order)"""
    width = R.WIDTH[name]
    limbs = words(n, width + segbits, _seed("segments", name, descending, segbits))
    seg = field(limbs, width, segbits).astype(np.int64)
    p = np.argsort(seg, kind="stable")
    seg = seg[p]
    raw = decode(field(limbs, 0, width)[p], name, descending)
    offsets = np.searchsorted(seg, np.arange((1 << segbits) + 1), side="left").astype(np.int64)
    return Plan([key_round(raw, name, descending), Round(seg.astype(np.uint64), 64, live=segbits, pad=True)],
                raw=raw, seg=seg, offsets=offsets, src=p, name=name, descending=descending)


# ---- steps and faults --------------------------------------------------------------------------------------------------------
def steps(plan, radix, shape):
    """[(round, shift, bits, reach)] in the order the call runs them; reach: where the digit would end unclamped (the
    last step of a clamped digit only).  Steps wholly above a round's live bits (constant) are left out."""
    out = []
    for k, rd in enumerate(plan.rounds):
        bits = rd.plan_bits(radix)
        for d in range(H.num_passes(radix, bits)):
            shift, b, lo, hi = H.plan_pass(radix, d, one_pass=shape == "one_pass", key_bits=bits)
            parts = [(shift, b)] if shape == "digit" or not lo else [(shift, lo), (shift + lo, hi)]
            for i, (s, w) in enumerate(parts):
                if s < rd.live:
                    out.append((k, s, w, shift + radix if i == len(parts) - 1 and b < radix else None))
    return out


def faults(plan, step):
    k, s, w, reach = step
    rd = plan.rounds[k]
    out = ["skip", "shift+1", "reverse"]
    if s and s + w <= rd.live:  # with a constant top bit, reading one bit lower reads what the steps below sorted
        out.append("shift-1")
    if w > 1:
        out.append("merge")
    if reach is not None and rd.above is not None and reach > rd.above:
        out.append("unclamped")
    if rd.raw is not None and (digit(rd, step, "raw") != digit(rd, step, None)).any():
        out.append("raw")  # where the raw bits are the order key's on every record, there is nothing to misread
    return out


def digit(rd, step, fault):
    """the digit the (faulty) step sorts by"""
    _, s, w, reach = step
    word = rd.raw if fault == "raw" else rd.word
    if fault == "skip":
        return np.zeros(len(word), dtype=np.uint64)
    s += {"shift+1": 1, "shift-1": -1}.get(fault, 0)
    if fault == "unclamped":
        w = reach - s
    d = word >> np.uint64(s) & _mask(w) if s < 64 else np.zeros(len(word), dtype=np.uint64)
    return d >> np.uint64(1) if fault == "merge" else d


class Checker:
    """fault detection on one plan; ranks below and above each bit position are cached"""

    def __init__(self, plan):
        self.plan, self.n = plan, plan.n
        self.correct = plan.order()
        self._below, self._above = {}, {}

    def below(self, k, s):
        """rank of every record in the stable sort by the rounds below k and the bits of round k below s"""
        if (k, s) not in self._below:
            keys = [r.key for r in self.plan.rounds[:k]] + ([self.plan.rounds[k].key & _mask(s)] if s else [])
            p = np.lexsort(keys) if keys else np.arange(self.n)
            rank = np.empty(self.n, dtype=np.int64)
            rank[p] = np.arange(self.n)
            self._below[k, s] = rank
        return self._below[k, s]

    def above(self, k, t):
        """dense rank of (bits of round k from t on, the rounds above k)"""
        if (k, t) not in self._above:
            rd = self.plan.rounds[k]
            keys = ([rd.key >> np.uint64(t)] if t < rd.bits else []) + [r.key for r in self.plan.rounds[k + 1:]]
            rank = np.zeros(self.n, dtype=np.int64)
            if keys:
                p = np.lexsort(keys)
                new = np.zeros(self.n, dtype=np.int64)
                new[1:] = np.any([np.diff(x[p]) != 0 for x in keys], axis=0)
                rank[p] = np.cumsum(new)
            self._above[k, t] = rank
        return self._above[k, t]

    def detected(self, step, fault):
        """does the fault change the output?"""
        k, s, w, _ = step
        nb = self.n.bit_length()
        tie = self.below(k, s)
        if fault == "reverse":
            tie = self.n - 1 - tie
        d = digit(self.plan.rounds[k], step, fault).astype(np.int64)
        key = (self.above(k, s + w) << (17 + nb)) | (d << nb) | tie
        return not bool((np.diff(key[self.correct]) > 0).all())

    def faulty_output(self, step, fault):
        """the faulty sort's output as input indices (for cross-checks; detected() does not sort)"""
        k, s, w, _ = step
        tie = self.below(k, s)
        if fault == "reverse":
            tie = self.n - 1 - tie
        return np.lexsort([tie, digit(self.plan.rounds[k], step, fault), self.above(k, s + w)])

    def undetected(self, radices=range(1, 17), shapes=SHAPES):
        """[(radix, shape, step index, step, fault)] whose fault leaves the output unchanged; each distinct (step,
        fault) is evaluated once"""
        seen, out = {}, []
        for radix in radices:
            for shape in shapes:
                for i, st in enumerate(steps(self.plan, radix, shape)):
                    for f in faults(self.plan, st):
                        key = (st[:3], f, st[3] if f == "unclamped" else None)
                        if key not in seen:
                            seen[key] = self.detected(st, f)
                        if not seen[key]:
                            out.append((radix, shape, i, st, f))
        return out


def lsd(plan, radix, shape, fault=None, at=None):
    """the LSD sort step by step (stable argsort per step), step `at` faulted: input indices in output order"""
    idx = np.arange(plan.n)
    for i, st in enumerate(steps(plan, radix, shape)):
        f = fault if i == at else None
        d = digit(plan.rounds[st[0]], st, f)[idx]
        if f == "reverse":  # ascending digits, equal digits in reversed order
            p = len(d) - 1 - np.argsort(d[::-1], kind="stable")
        else:
            p = np.argsort(d, kind="stable")
        idx = idx[p]
    return idx
