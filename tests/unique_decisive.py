"""Inputs on which every step of lsb_unique_device decides the output, and the fault model that proves it.

A unique kernel hides a fault wherever two neighbouring groups differ in many bits or in several rounds at once: a head
test that ignores one bit still sees the others.  The inputs here are built as a sequence of groups in the mode's order
(lexsort order in sorted mode, input order in consecutive mode) whose neighbours differ, as often as possible, in one bit
of one column only, and whose group starts sit on the positions where the kernels change how they find the neighbour.

Keys.  Every column is walked as a chain of order-key words whose neighbours differ in one bit each, with the columns
below it held at their first key; the columns below are walked the same way at the chain's last word, and so on down to
column 0.  A chain word is a reachable order key (one some bit pattern encodes to: decisive.decode / encode), so floats
skip the NaN words but one and the word of -0.0.  A float column's chain runs up from the word of +0.0 and then from its
lowest infinity up to +0.0, and visits the NaN word: groups at those two words hold twins (NaNs of both signs and
several payloads, -0.0 and +0.0), equal keys with different bits.

Sorted mode cannot hold a single-bit neighbour at every bit of every column.  Two such neighbours in one column, with
the same columns above it, span disjoint ranges of that column's words, and together the W bits span 2^W - 1 words.
A float has fewer reachable words, so one bit of a float column is left over; it is placed under another word of a
float column above it, which has words to spare, and is unreachable when only integer columns (or none) are above it.
`Block.lost` lists those bits, and the fault checker skips exactly them.  Consecutive mode has neighbours in input order
and places the left-over bits as plain pairs, so it misses none.

Positions.  Run lengths put a round-r-only group start at a lane-0 position (p % 32 == 0) and another at p % 32 == 31
with a run of two or more after it, for every round; at odd tiles the positions 2048 t - 1, 2048 t and 2048 t + 1 all
start groups, at even tiles none of them does.  Large inputs (`large_lengths`) put group starts decided by each earlier
round alone, and non-starts, on the grid-stride boundaries of unique_flag_kernel and on their IO_U multiples.

Faults.  `Model` restates the kernels in numpy: head flags per round (unique_flag_kernel for earlier rounds,
unique_tile_kernel for the last), per-tile counts, their exclusive scan, then index / inverse / ends / counts.  `faults`
lists one-line faults of those steps; `Checker.undetected` returns the ones that leave (U, index, inverse, counts) of an
input unchanged.  A fault that only changes head flags changes the output exactly when it changes some flag, so those
are checked on the flags.
"""
import zlib

import numpy as np

import decisive as D
import lexsort_ref as R
from distributed_lsb_b200 import hostlogic as H

TILE = 2048          # positions of a unique_tile_kernel CTA (UNIQUE_THREADS x UNIQUE_ITEMS)
WARP = 32
IO_THREADS = 256
IO_U = 4
IO_CTAS_PER_SM = 4
SENTINEL = -7
MIN_GROUPS = 128
LAST_RUN = 40
BLOCK_N = 6 * TILE + 77                # the GPU inputs at every radix
LARGE_N = (1 << 21) + 77               # at least three IO_U steps of the flag kernel's grid stride up to 170 SMs
FLOATS = {"float64": 52, "float32": 23, "float16": 10, "bfloat16": 7}  # mantissa bits

# (names, descending), least significant column first.  Every type in both directions sits in an earlier round in
# one mix and in the last round in another; there are 1, 2 and 3 rounds, and rounds of 1, 2, 3 and 4 columns in both
# kernels.  Each mix also runs with every direction flipped.
MIXES = [
    (("float64",), (False,)),
    (("bfloat16",), (True,)),
    (("uint64", "int64", "float64"), (False, True, True)),
    (("float64", "uint64", "int64"), (False, True, False)),
    (("int64", "float64", "uint64"), (False, True, True)),
    (("float32", "int32", "uint64"), (False, True, False)),
    (("uint16", "int16", "float16", "bfloat16", "uint32", "float16", "bfloat16", "int64"),
     (False, True, False, True, True, True, False, True)),
    (("int32", "float32", "uint32", "int16", "uint16"), (False, True, False, False, True)),
    (("uint32", "int16", "uint16", "uint16", "int16", "float16", "bfloat16"), (False, False, True, False, True, False, True)),
    (("uint64", "uint32", "float16", "bfloat16"), (True, True, True, False)),
    (("float64", "int32", "float32"), (True, True, False)),
    (("uint16", "uint16", "int16", "float16", "int32", "float32"), (True, False, False, True, False, True)),
]


def cases():
    """(mix, flipped) -> (names, descending)"""
    return {(m, f): (names, tuple(d != f for d in desc)) for m, (names, desc) in enumerate(MIXES) for f in (False, True)}


def rounds(names):
    """lexsort's rounds [(first, ncols, bits, passes at radix 16)]; which columns share a round does not depend on the
    radix"""
    return H.lexsort_rounds([R.WIDTH[x] for x in names], 16)


def shifts(names):
    """(round, shift in the round's word) of every column"""
    out = []
    for r, (first, ncols, _, _) in enumerate(rounds(names)):
        at = 0
        for c in range(first, first + ncols):
            out.append((r, at))
            at += R.WIDTH[names[c]]
    return out


# ---- words ---------------------------------------------------------------------------------------------------------------
def _reachable(name, desc, *ws):
    a = np.array(ws, dtype=np.uint64)
    return bool((D.encode(D.decode(a, name, desc), name, desc) == a).all())


def _word(name, desc, raw):
    return int(D.encode(np.array([raw], dtype=R.UINT[R.WIDTH[name]]), name, desc)[0])


def special_raws(name):
    """(+0.0, the infinities, NaNs of both signs and several payloads, -0.0) of a float type as bit patterns"""
    w, m = R.WIDTH[name], FLOATS[name]
    sign, exp = 1 << (w - 1), ((1 << (w - 1)) - 1) ^ ((1 << m) - 1)
    nans = [exp | 1 << (m - 1), sign | exp | 1 << (m - 1), exp | 1, sign | exp | ((1 << m) - 1), exp | (0x55555555 & ((1 << m) - 1))]
    return {"zero": 0, "negzero": sign, "inf": exp, "neginf": sign | exp, "nans": nans}


def _greedy(name, desc, bits, lo, hi):
    """single-bit pairs (x, b) in increasing order with disjoint spans inside [lo, hi]: bit b of x clear, x and x + 2^b
    reachable; bits ascending, each placed at the lowest word it fits"""
    pairs, cur = [], lo
    for b in sorted(bits):
        s = 1 << b
        x = cur if not cur & s else (cur | (2 * s - 1)) + 1
        for cand in (x, x + 1, x + 2 * s, x + 2 * s + 1):
            if not cand & s and cand + s <= hi and _reachable(name, desc, cand, cand + s):
                pairs.append((cand, b))
                cur = cand + s
                break
    return pairs


def chain(name, desc, bits):
    """(words, covered bits): increasing reachable words of a column, neighbours one bit apart wherever a bit of `bits`
    is placed; floats also visit +0.0 and the NaN word (twins)"""
    if name not in FLOATS:
        pairs = _greedy(name, desc, bits, *_span(name, desc))
        words = sorted({w for x, b in pairs for w in (x, x + (1 << b))}) or [0]
        return words, {b for _, b in pairs}
    sp = special_raws(name)
    zero, nan = _word(name, desc, sp["zero"]), _word(name, desc, sp["nans"][0])
    lo, hi = _span(name, desc)
    up = _greedy(name, desc, bits, zero, hi)
    pairs = _greedy(name, desc, set(bits) - {b for _, b in up}, lo, zero) + up
    full = _greedy(name, desc, bits, lo, hi)  # one sweep over all the words: what a bit left over alone needs
    if len(full) > len(pairs):
        pairs = full
    inside = any(x < zero < x + (1 << b) for x, b in pairs)
    words = sorted({w for x, b in pairs for w in (x, x + (1 << b))} | (set() if inside else {zero}))
    return ([nan] + words if nan < lo else words), {b for _, b in pairs}


def _span(name, desc):
    """the lowest and highest reachable word but NaN"""
    if name not in FLOATS:
        return 0, (1 << R.WIDTH[name]) - 1
    sp = special_raws(name)
    return tuple(sorted((_word(name, desc, sp["inf"]), _word(name, desc, sp["neginf"]))))


def _next_free(name, desc, after, below):
    """the lowest reachable word in (after, below), or None"""
    for w in range(after + 1, min(after + 4097, below)):
        if _reachable(name, desc, w):
            return w
    return None


def _sweep(names, desc, sig, need):
    """keys (tuples of order-key words over the columns `sig`, most significant first), strictly increasing in lexsort
    order; removes the bits it places from need[c]"""
    if not sig:
        return [()]
    c, rest = sig[0], sig[1:]
    name, d = names[c], desc[c]
    words, got = chain(name, d, need[c])
    need[c] = need[c] - got
    sub = _sweep(names, desc, rest, need)
    out = []

    def emit(k):
        if not out or out[-1] != k:
            assert not out or out[-1] < k, (out[-1], k)
            out.append(k)

    nan = _word(name, d, special_raws(name)["nans"][0]) if name in FLOATS else None
    for w in words:
        emit((w,) + sub[0])
    for s in sub:
        emit((words[-1],) + s)
    # bits the columns below could not place under this word: again under the next free words of this column
    v, top = words[-1], (nan if nan is not None and nan > words[-1] else 1 << R.WIDTH[name])
    while any(need[x] for x in rest):
        before = sum(len(need[x]) for x in rest)
        v = _next_free(name, d, v, top)
        if v is None:
            break
        for s in _sweep(names, desc, rest, need):
            emit((v,) + s)
        if sum(len(need[x]) for x in rest) == before:
            break
    if nan is not None and nan > words[-1]:  # a NaN word above the infinities comes last
        emit((nan,) + sub[0])
    return out


def _pad(keys, names, desc):
    """at least MIN_GROUPS keys: more words of the primary column after the last key (before a NaN key that ends the
    sequence), so that short sequences still start groups in every tile"""
    c = len(names) - 1
    name, d = names[c], desc[c]
    nan = _word(name, d, special_raws(name)["nans"][0]) if name in FLOATS else None
    tail = [keys.pop()] if nan is not None and keys[-1][c] == nan and len(keys) > 1 else []
    while len(keys) + len(tail) < MIN_GROUPS:
        v = _next_free(name, d, keys[-1][c], nan if tail else 1 << R.WIDTH[name])
        if v is None:  # an integer chain ends at the column's top word
            break
        keys.append(keys[-1][:c] + (v,))
    return keys + tail


class Block:
    """the group sequence of one mix in one mode: keys[g] the order-key words of group g (column order), `lost` the
    (column, bit) pairs no single-bit neighbour covers (sorted mode only)"""

    def __init__(self, names, desc, consecutive):
        self.names, self.desc, self.consecutive = tuple(names), tuple(desc), consecutive
        K = len(names)
        need = {c: set(range(R.WIDTH[names[c]])) for c in range(K)}
        keys = [k[::-1] for k in _sweep(names, desc, list(range(K - 1, -1, -1)), need)]
        left = sorted((c, b) for c in need for b in need[c])
        if consecutive:  # plain pairs at the end, then back: A B A
            for c, b in left:
                (x, _), = _greedy(names[c], desc[c], [b], *_span(names[c], desc[c]))
                a = list(keys[-1])
                a[c] = x
                bb = list(a)
                bb[c] = x + (1 << b)
                keys += [tuple(a), tuple(bb), tuple(a)]
            left = []
        self.keys = _pad([k for i, k in enumerate(keys) if i == 0 or k != keys[i - 1]], names, desc)
        self.lost = left

    def twins(self):
        """the groups whose key holds +0.0 or the NaN word in a float column"""
        special = {c: {_word(x, d, special_raws(x)["zero"]), _word(x, d, special_raws(x)["nans"][0])}
                   for c, (x, d) in enumerate(zip(self.names, self.desc)) if x in FLOATS}
        return {g for g, k in enumerate(self.keys) if any(k[c] in w for c, w in special.items())}

    def kinds(self):
        """for every group start g >= 1: the set of rounds whose words differ from group g - 1's"""
        sh = shifts(self.names)
        out = [None]
        for a, b in zip(self.keys, self.keys[1:]):
            out.append({sh[c][0] for c in range(len(a)) if a[c] != b[c]})
        return out


def _seed(*what):
    return zlib.crc32(repr(what).encode())


# ---- run lengths ------------------------------------------------------------------------------------------------------------
def block_lengths(block, n=BLOCK_N):
    """run lengths summing to n: a round-r-only start at p % 32 == 0 and one at p % 32 == 31 followed by a run >= 2, for
    every round r, the other starts on residues mod 32 in turn; at tile t (t >= 1) the starts 2048 t - 1, 2048 t and
    2048 t + 1 are all group starts (t odd) or none (t even); the last group starts LAST_RUN before the end"""
    kinds = block.kinds()
    G = len(kinds)
    rng = np.random.default_rng(_seed("lengths", block.names, block.desc, block.consecutive))
    nr = len(rounds(block.names))
    want = {0: set(range(nr)), 31: set(range(nr))}
    forced = {t * TILE + o for t in range(1, n // TILE + 1, 2) for o in (-1, 0, 1)}
    banned = {t * TILE + o for t in range(2, n // TILE + 1, 2) for o in (-1, 0, 1)}
    twins = block.twins()
    lengths, pos, atleast2, turn = [], 0, False, 0
    for g in range(G - 1):
        atleast2 = atleast2 or g in twins
        k = kinds[g + 1]
        single = next(iter(k)) if len(k) == 1 else None
        target = 0 if single in want[0] else 31 if single in want[31] else None
        mean = max(1, (n - LAST_RUN - pos) // (G - 1 - g))
        if target is None:
            target, turn = turn, (turn + 7) % WARP
            single = None
        L = (target - pos) % WARP or WARP
        L += WARP * int(rng.integers(0, max(1, 2 * mean // WARP)))
        if atleast2:
            L = max(L, 2)
        f = min((x for x in forced if x > pos), default=None)
        if f is not None and pos + L > f:
            L = f - pos
        while pos + L in banned:
            L += 1
        L = max(1, min(L, n - LAST_RUN - pos - (G - 2 - g)))
        if g == G - 2:
            L = n - LAST_RUN - pos
        end = pos + L
        if single is not None and end % WARP == target:
            want[target].discard(single)
        atleast2 = single is not None and target == 31 and end % WARP == 31
        lengths.append(L)
        pos += L
    lengths.append(n - pos)
    assert pos == n - LAST_RUN and min(lengths) >= 1 and not want[0] and not want[31], (want, pos)
    return np.array(lengths, dtype=np.int64)


def grid_stride(sms, n):
    """unique_flag_kernel's grid stride on a card with `sms` SMs: io_grid(n) x IO_THREADS"""
    return min(sms * IO_CTAS_PER_SM, -(-n // IO_THREADS)) * IO_THREADS


def grid_targets(block, stride, n):
    """{position: round whose flag alone starts a group there, or None for a non-start} on the grid-stride boundaries
    k * stride (k = 1, 2, 5) and IO_U-step boundaries (k = 4, 8, 12) of the flag kernel, for the earlier rounds in the
    order their single-round starts come in the group sequence"""
    kinds = block.kinds()
    nr = len(rounds(block.names))
    seen = []
    for k in kinds[1:]:
        if len(k) == 1 and next(iter(k)) < nr - 1 and next(iter(k)) not in seen:
            seen.append(next(iter(k)))
    e = seen + [None] * (2 - len(seen))
    plan = {1: e[0], 2: None, 4: e[0], 5: e[1], 8: e[1], 12: None}
    return {k * stride: r for k, r in plan.items() if k * stride < n}


def large_lengths(block, stride, n=LARGE_N):
    """run lengths summing to n with grid_targets(block, stride, n) in place: a start of the named round alone exactly
    on each such position, no start on the others"""
    kinds = block.kinds()
    G = len(kinds)
    targets = grid_targets(block, stride, n)
    heads = sorted((p, r) for p, r in targets.items() if r is not None)
    banned = {p for p, r in targets.items() if r is None}
    starts, g = [0], 0  # starts[g] of group g
    for p, r in heads:
        j = next(j for j in range(g + 1, G) if kinds[j] == {r})
        assert j - g <= p - starts[-1] and G - j >= 2
        starts += list(np.linspace(starts[-1], p, j - g + 1).astype(np.int64)[1:])
        g = j
    starts += list(np.linspace(starts[-1], n, G - g + 1).astype(np.int64)[1:-1])
    starts = np.array(starts + [n], dtype=np.int64)
    for i in range(1, G):
        while int(starts[i]) in banned:
            starts[i] += 1
    lengths = np.diff(starts)
    assert len(lengths) == G and lengths.min() >= 1 and lengths.sum() == n
    return lengths


# ---- elements ---------------------------------------------------------------------------------------------------------------
def elements(block, lengths, seed=0):
    """bit-pattern columns (least significant first) of the input: group g repeated lengths[g] times, in input order
    (consecutive) or shuffled (sorted); the elements of a group at a float column's +0.0 or NaN word take the twins'
    patterns in turn"""
    names, desc = block.names, block.desc
    n = int(lengths.sum())
    rng = np.random.default_rng(_seed("elements", names, desc, block.consecutive, n, seed))
    g = np.repeat(np.arange(len(block.keys)), lengths)
    cols = []
    for c, (x, d) in enumerate(zip(names, desc)):
        words = np.array([k[c] for k in block.keys], dtype=np.uint64)
        raw = D.decode(words, x, d)[g]
        if x in FLOATS:
            sp = special_raws(x)
            for which, pats in (("zero", [sp["zero"], sp["negzero"]]), ("nans", sp["nans"])):
                at = np.flatnonzero(words[g] == np.uint64(_word(x, d, sp[which] if which == "zero" else sp["nans"][0])))
                pats = np.array(pats, dtype=raw.dtype)
                raw[at] = pats[np.arange(len(at)) % len(pats)]
        cols.append(raw)
    if not block.consecutive:
        p = rng.permutation(n)
        cols = [x[p] for x in cols]
    return cols


def block_input(mix, flipped, consecutive):
    """the proven input of BLOCK_N elements the GPU module runs at every radix"""
    names, desc = cases()[mix, flipped]
    b = Block(names, desc, consecutive)
    return b, elements(b, block_lengths(b))


def large_input(mix, flipped, consecutive, sms):
    names, desc = cases()[mix, flipped]
    b = Block(names, desc, consecutive)
    stride = grid_stride(sms, LARGE_N)
    return b, elements(b, large_lengths(b, stride), seed=1), stride


# ---- the kernels in numpy, and their faults ------------------------------------------------------------------------------------
class Model:
    """lsb_unique_device on bit-pattern columns: round words from order keys (lexsort_pack_kernel's), lexsort order
    (sorted) or input order, head flags, tile counts and scan, outputs"""

    def __init__(self, cols, names, desc, consecutive, stride=None):
        self.names, self.desc, self.consecutive, self.stride = tuple(names), tuple(desc), consecutive, stride
        self.n = n = len(cols[0])
        self.rounds = rounds(names)
        sh = shifts(names)
        self.cols = [(r, s, D.encode(b, x, d), np.asarray(b).astype(np.uint64), x)
                     for (r, s), b, x, d in zip(sh, cols, names, desc)]
        words = [np.zeros(n, dtype=np.uint64) for _ in self.rounds]
        for r, s, ok, _, _ in self.cols:
            words[r] |= ok << np.uint64(s)
        self.order = np.arange(n) if consecutive else np.lexsort(words)
        self.W = [w[self.order] for w in words]
        self.pos = np.arange(n)
        self.correct_heads = self.heads()
        self.correct = self.outputs(self.correct_heads)

    def _flags(self, r, f):
        w = self.W[r]
        if f[0] == "mask" and f[1] == r:
            w = w & ~np.uint64(1 << f[2])
        if f[0] == "raw" and f[1] == r:
            _, s, ok, raw, _ = self.cols[f[2]]
            w = w ^ ((ok ^ raw) << np.uint64(s))[self.order]
        prev = np.empty_like(w)
        prev[1:] = w[:-1]
        prev[0] = w[0]
        lane0 = (self.pos % WARP == 0) & (self.pos > 0)
        if f[0] == "lane0_prev2" and f[1] == r:
            at = lane0 & (self.pos >= 2)
            prev[at] = w[self.pos[at] - 2]
        if f[0] == "lane0_self" and f[1] == r:
            prev[lane0] = w[lane0]
        d = w != prev
        d[0] = False
        if f[0] == "grid" and f[1] == r:
            d[(self.pos % f[2] == 0) & (self.pos > 0)] = f[3]
        return d

    def heads(self, f=("none",)):
        last = len(self.rounds) - 1
        diff = np.zeros(self.n, dtype=bool)
        for r in range(last):
            d = self._flags(r, f)
            if f == ("drop", r):
                continue
            diff = d if (r == 0 or f == ("write", r)) else diff | d
        h = self._flags(last, f) | diff
        h[0] = True
        if f[0] == "tile_start":
            h[(self.pos % TILE == 0) & (self.pos > 0)] = f[1]
        return h

    def outputs(self, h, f=("none",)):
        """(U, index, inverse, counts): arrays of n, SENTINEL where nothing is written"""
        n, T = self.n, -(-self.n // TILE)
        t = self.pos // TILE
        totals = np.bincount(t, weights=h, minlength=T).astype(np.int64)
        base = np.concatenate([[0], np.cumsum(totals)])
        tb = base[:T].copy()
        if f[0] == "tile_base":
            tb[f[1]] = base[f[1] + 1]
        c = np.cumsum(h)
        before = np.concatenate([[0], c[TILE - 1::TILE]])[:T]
        r = tb[t] + c - before[t] - 1
        u = int(tb[T - 1] + totals[T - 1])
        index, inverse, ends, counts = (np.full(n, SENTINEL, dtype=np.int64) for _ in range(4))
        hp = np.flatnonzero(h)
        ok = (r[hp] >= 0) & (r[hp] < n)
        src = hp
        if f[0] == "index_last":  # the last position of every group
            src = np.append(hp[1:], n) - 1
        index[r[hp][ok]] = self.order[src][ok]
        e = hp + (f[1] if f[0] == "ends" else 0)
        sel = ok & (r[hp] >= 1)
        ends[r[hp][sel] - 1] = e[sel]
        inverse[self.pos if f[0] == "inverse_sorted" else self.order] = r
        rr = np.arange(min(max(u, 0), n))
        hi = np.where(rr + 1 < u, ends[np.minimum(rr, n - 1)], n - (f[0] == "count_last"))
        counts[rr] = hi - np.where(rr > 0, ends[np.maximum(rr - 1, 0)], 0)
        return u, index, inverse, counts

    def result(self):
        u, index, inverse, counts = self.correct
        return u, index[:u], inverse, counts[:u]


HEAD_FAULTS = ("mask", "raw", "lane0_prev2", "lane0_self", "grid", "drop", "write", "tile_start")


def faults(model, lost=()):
    """every fault of the model on this input's geometry; mask faults of `lost` (column, bit) are left out"""
    sh = shifts(model.names)
    skip = {(sh[c][0], sh[c][1] + b) for c, b in lost}
    last = len(model.rounds) - 1
    out = []
    for r, (_, _, bits, _) in enumerate(model.rounds):
        out += [("mask", r, b) for b in range(bits) if (r, b) not in skip]
        out += [("lane0_prev2", r), ("lane0_self", r)]
        out += [("raw", r, c) for c, (rc, _, _, _, x) in enumerate(model.cols) if rc == r and x in FLOATS]
        if r < last:
            out.append(("drop", r))
            if r > 0:
                out.append(("write", r))
            if model.stride:
                out += [("grid", r, m, v) for m in (model.stride, IO_U * model.stride) for v in (True, False)]
    out += [("tile_start", True), ("tile_start", False)]
    out += [("tile_base", t) for t in range(-(-model.n // TILE))]
    if not model.consecutive:
        out.append(("inverse_sorted",))
    out += [("index_last",), ("count_last",), ("ends", 1), ("ends", -1)]
    return out


class Checker:
    def __init__(self, model):
        self.m = model

    def detected(self, f):
        m = self.m
        h = m.heads(f) if f[0] in HEAD_FAULTS else m.correct_heads
        if f[0] in HEAD_FAULTS:
            return not np.array_equal(h, m.correct_heads)
        got = m.outputs(h, f)
        return got[0] != m.correct[0] or not all(np.array_equal(a, b) for a, b in zip(got[1:], m.correct[1:]))

    def detected_full(self, f):
        """detected() through the whole output, head faults too"""
        m = self.m
        got = m.outputs(m.heads(f) if f[0] in HEAD_FAULTS else m.correct_heads, f)
        return got[0] != m.correct[0] or not all(np.array_equal(a, b) for a, b in zip(got[1:], m.correct[1:]))

    def undetected(self, fs):
        return [f for f in fs if not self.detected(f)]

    def mask_undetected(self):
        """(round, bit) of every mask fault the input hides: a start p shows bit b of round r only when round r is the
        only round whose words differ from p - 1's and they differ in bit b alone"""
        m = self.m
        x = [np.concatenate([[np.uint64(0)], w[1:] ^ w[:-1]]) for w in m.W]
        nz = np.array([v != 0 for v in x])
        seen = set()
        for r, v in enumerate(x):
            only = nz[r] & (nz.sum(axis=0) == 1) & ((v & (v - np.uint64(1))) == 0)
            for val in np.unique(v[only]):
                seen.add((r, int(val).bit_length() - 1))
        return [(r, b) for r, (_, _, bits, _) in enumerate(m.rounds) for b in range(bits) if (r, b) not in seen]
