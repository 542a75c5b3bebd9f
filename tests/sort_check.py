"""An independent checker of stable sorts for the tests, in plain torch on any device, for sizes past 2^31.

check_sort decides whether an output is exactly the stable sort by (segment, key) of an input, in O(n) work and about
n bytes of whole-length memory (one bool per element); the rest runs in chunks.  It is written from the key orders of
include/lsbsort.h and imports nothing from the library: the library's own verify() is the code under test, not a
reference.  Keys are compared as int64 bit patterns (torch's uint64 support on CUDA is partial), so NaN payloads and
-0.0 count.

The key makers build seeded inputs on the device in chunks from a counter hash (splitmix64), so an input of 2^31 keys
needs no host memory and no temporary of its own size.
"""
import torch

INT64_MIN = -(1 << 63)
INT64_MAX = (1 << 63) - 1
I64, F64, DESC = 16, 32, 64  # LSB_FLAG_KEY_I64, LSB_FLAG_KEY_F64, LSB_FLAG_DESCENDING of include/lsbsort.h
CHUNK = 1 << 27
F64_INF = 0x7FF0000000000000
GATHER_C = 0x5DEECE66DA3B9F17  # vals_in[i] = (i << 16) ^ GATHER_C; low 16 bits 0x9F17 != 0
CONTEXT = 3  # elements shown on either side of a failing position


def _s64(u):
    """a uint64 constant as the int64 of the same bits"""
    return u - (1 << 64) if u >= 1 << 63 else u


def _i64(t):
    return t if t.dtype == torch.int64 else t.view(torch.int64)


def order_key(bits, korder):
    """int64 bit patterns of keys -> int64 whose ascending order is the order `korder` (I64 / F64 / DESC) sorts by:
    uint64 b ^ INT64_MIN; int64 b; float64 -0.0 read as +0.0, every NaN INT64_MAX, otherwise b ^ ((b >> 63) & INT64_MAX)
    (negative doubles reversed); descending the bitwise NOT of the ascending key"""
    b = _i64(bits)
    if korder & F64:
        b = torch.where(b == INT64_MIN, torch.zeros_like(b), b)
        k = b ^ ((b >> 63) & INT64_MAX)
        k = torch.where((b & INT64_MAX) > F64_INF, torch.full_like(b, INT64_MAX), k)
    elif korder & I64:
        k = b
    else:
        k = b ^ INT64_MIN
    return ~k if korder & DESC else k


def segment_of(offsets, pos):
    """segment of every position in `pos`: searchsorted(offsets, pos, right=True) - 1 (empty segments own none)"""
    return torch.searchsorted(offsets, pos, right=True) - 1


# ---- decoders: the global input index of every output position, from what a sort returns ---------------------------------
class GlobalIndex:
    """vals_out holds the global input index (sort_device or sort_segments without vals)"""
    def __init__(self, idx):
        self.t = _i64(idx)

    def __call__(self, lo, hi):
        return self.t[lo:hi], None


class LocalIndex:
    """vals_out holds the index within the segment: idx = local + offsets[seg(j)]"""
    def __init__(self, local, offsets):
        self.t, self.offsets = _i64(local), offsets

    def __call__(self, lo, hi):
        pos = torch.arange(lo, hi, dtype=torch.int64, device=self.t.device)
        return self.t[lo:hi] + self.offsets[segment_of(self.offsets, pos)], None


def gather_vals(n, device, dtype=torch.int64):
    """vals_in[i] = (i << 16) ^ GATHER_C, invertible; as int64 or as the float64 of the same bits"""
    v = torch.empty(n, dtype=torch.int64, device=device)
    for lo in range(0, n, CHUNK):
        v[lo:lo + CHUNK] = (torch.arange(lo, min(lo + CHUNK, n), dtype=torch.int64, device=device) << 16) ^ GATHER_C
    return v if dtype == torch.int64 else v.view(dtype)


class GatheredVals:
    """vals_out holds gather_vals()[idx]: idx = (v ^ GATHER_C) >> 16, and the low 16 bits must be GATHER_C's"""
    def __init__(self, vals):
        self.t = _i64(vals)

    def __call__(self, lo, hi):
        x = self.t[lo:hi] ^ GATHER_C
        return x >> 16, (x & 0xFFFF) == 0


# ---- the checker ------------------------------------------------------------------------------------------------------------
def _window(j, n, keys_in, keys_out, decode, korder, offsets, note=""):
    """positions j - CONTEXT .. j + CONTEXT: output key bits, order key, decoded index, input key there, segments"""
    lo, hi = max(0, j - CONTEXT), min(n, j + CONTEXT + 1)
    idx, _ = decode(lo, hi)
    ko = _i64(keys_out)[lo:hi]
    ok = order_key(ko, korder)
    valid = (idx >= 0) & (idx < n)
    kin = torch.where(valid, _i64(keys_in)[torch.where(valid, idx, 0)], 0)
    pos = torch.arange(lo, hi, dtype=torch.int64, device=idx.device)
    rows = [f"{'pos':>12} {'keys_out bits':>18} {'order_key':>21} {'idx':>12} {'keys_in[idx] bits':>18}"
            + ("  seg(pos) seg(idx)" if offsets is not None else "")]
    seg_p = segment_of(offsets, pos).tolist() if offsets is not None else None
    seg_i = segment_of(offsets, torch.where(valid, idx, 0)).tolist() if offsets is not None else None
    for r, (p, k, o, i, ki, v) in enumerate(zip(pos.tolist(), ko.tolist(), ok.tolist(), idx.tolist(), kin.tolist(),
                                                 valid.tolist())):
        row = (f"{'>' if p == j else ' '}{p:>11} {k & (2**64 - 1):018x} {o:>21} {i:>12} "
               + (f"{ki & (2**64 - 1):018x}" if v else f"{'out of range':>18}"))
        if offsets is not None:
            row += f"  {seg_p[r]:>8} {seg_i[r] if v else '-':>8}"
        rows.append(row)
    return note + "\n" + "\n".join(rows)


def _first(mask):
    """index of the first True of a bool tensor, or None"""
    hit = mask.nonzero()
    return int(hit[0, 0]) if len(hit) else None


def check_sort(keys_in, keys_out, idx, korder, offsets=None, chunk=CHUNK):
    """None if keys_out, with the input indices `idx`, is exactly the stable sort of keys_in by (segment, order_key) --
    one segment without `offsets`, else segment s = positions [offsets[s], offsets[s+1]) of input and output.  Otherwise
    a message naming the first failing position of the first failing check, with the elements around it.

    keys_in / keys_out: 1-D tensors of 8-byte keys (any dtype, read as bits).  idx: an int64 tensor of global input
    indices, or a decoder (LocalIndex, GatheredVals).  The checks, in this order:
      1. every idx in [0, n) (and a gathered value decodes: its low 16 bits are GATHER_C's) -- before any indexing;
      2. idx is a permutation: a bool[n] set through idx is all True;
      3. keys_out[j] == keys_in[idx[j]] bit for bit;
      4. inside every output segment, (order_key(keys_out), idx) strictly increases;
      5. seg(idx[j]) == seg(j): every element stays in its segment.
    1 and 2 run over the whole array first; 3-5 then run chunk by chunk, in order within each chunk."""
    decode = idx if callable(idx) else GlobalIndex(idx)
    n = keys_in.numel()
    if keys_out.numel() != n:
        return f"keys_out has {keys_out.numel()} elements, keys_in {n}"
    kin, kout = _i64(keys_in), _i64(keys_out)
    dev = kin.device
    if offsets is not None:
        offsets = _i64(offsets)
        if offsets.numel() < 2 or int(offsets[0]) != 0 or int(offsets[-1]) != n or bool((offsets[1:] < offsets[:-1]).any()):
            return f"offsets must rise from 0 to n = {n}"
    window = lambda j, note: _window(j, n, keys_in, keys_out, decode, korder, offsets, note)  # noqa: E731

    # 1 and 2: the range first, so that no gather or scatter below can read out of bounds
    seen = torch.zeros(n, dtype=torch.bool, device=dev)
    for lo in range(0, n, chunk):
        hi = min(lo + chunk, n)
        i, decodes = decode(lo, hi)
        bad = (i < 0) | (i >= n)
        if decodes is not None:
            bad |= ~decodes
        j = _first(bad)
        if j is not None:
            return window(lo + j, f"check 1: idx at position {lo + j} is out of [0, {n}) or does not decode")
        seen[i] = True
    if not bool(seen.all()):
        missing = _first(~seen)
        seen.zero_()  # the first position whose index an earlier position already holds
        for lo in range(0, n, chunk):
            hi = min(lo + chunk, n)
            i, _ = decode(lo, hi)
            dup = seen[i]
            s, order = torch.sort(i, stable=True)
            again = torch.zeros_like(dup)
            again[order[1:]] = s[1:] == s[:-1]
            j = _first(dup | again)
            if j is not None:
                return window(lo + j, f"check 2: idx is not a permutation: input index {missing} is missing, and "
                                      f"position {lo + j} repeats input index {int(i[j])}")
            seen[i] = True
        return f"check 2: idx is not a permutation: input index {missing} is missing"
    del seen

    for lo in range(0, n, chunk):
        hi = min(lo + chunk, n)
        ext = min(hi + 1, n)  # one element of overlap for the pairs (j, j + 1)
        i, _ = decode(lo, ext)
        ko = kout[lo:ext]
        j = _first(ko[:hi - lo] != kin[i[:hi - lo]])
        if j is not None:
            return window(lo + j, f"check 3: keys_out[{lo + j}] is not keys_in[idx[{lo + j}]] bit for bit")
        ok = order_key(ko, korder)
        rising = (ok[:-1] < ok[1:]) | ((ok[:-1] == ok[1:]) & (i[:-1] < i[1:]))
        if offsets is not None:
            seg = segment_of(offsets, torch.arange(lo, ext, dtype=torch.int64, device=dev))
            rising |= seg[:-1] != seg[1:]  # a pair across a segment boundary is not ordered
        j = _first(~rising)
        if j is not None:
            return window(lo + j, f"check 4: (order_key, idx) does not rise from position {lo + j} to {lo + j + 1}")
        if offsets is not None:
            j = _first(segment_of(offsets, i[:hi - lo]) != seg[:hi - lo])
            if j is not None:
                return window(lo + j, f"check 5: position {lo + j} holds input index {int(i[j])} of another segment")
    return None


# ---- seeded key makers on the device -----------------------------------------------------------------------------------
def splitmix64(x):
    """splitmix64's finaliser of int64 counters, in wrapping int64 arithmetic with logical right shifts"""
    z = x * _s64(0x9E3779B97F4A7C15) + _s64(0x9E3779B97F4A7C15)
    z = (z ^ ((z >> 30) & ((1 << 34) - 1))) * _s64(0xBF58476D1CE4E5B9)
    z = (z ^ ((z >> 27) & ((1 << 37) - 1))) * _s64(0x94D049BB133111EB)
    return z ^ ((z >> 31) & ((1 << 33) - 1))


def _fill(n, device, seed, f, out=None):
    """int64[n] with out[i] = f(splitmix64(i + seed * 2^40), i), made chunk by chunk (into `out`, any 8-byte dtype,
    when given)"""
    out = torch.empty(n, dtype=torch.int64, device=device) if out is None else _i64(out)
    for lo in range(0, n, CHUNK):
        i = torch.arange(lo, min(lo + CHUNK, n), dtype=torch.int64, device=device)
        out[lo:lo + CHUNK] = f(splitmix64(i + (seed << 40)), i)
    return out


def uniform_keys(n, device, seed=0, out=None):
    """bit patterns uniform over all 64 bits"""
    return _fill(n, device, seed, lambda h, i: h, out)


HOT_KEY = _s64(0xC3A5C85C97CB3127)
COLD_SHIFT = 12


def heavy_hitter_keys(n, device, seed=0, out=None):
    """HOT_KEY at all but one position in 2^COLD_SHIFT (99.976 %), uniform keys elsewhere: at n = 2^31 + 2^20 + 7 the
    hot key alone is more than 2^31 elements, so one bin of every pass holds that many"""
    return _fill(n, device, seed, lambda h, i: torch.where(
        (splitmix64(h) & ((1 << COLD_SHIFT) - 1)) == 0, h, torch.full_like(h, HOT_KEY)), out)


SPECIAL_BITS = [_s64(b) for b in (  # +-0, +-inf, NaNs of both signs with payloads, subnormals, extremes, +-1
    0x0000000000000000, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000, 0x7FF8000000000000,
    0xFFF8000000000000, 0x7FF8000000000123, 0xFFFC0000000ABCDE, 0x7FF0000000000001, 0xFFF0000000000001,
    0x7FF4000000000042, 0x0000000000000001, 0x8000000000000001, 0x7FEFFFFFFFFFFFFF, 0xFFEFFFFFFFFFFFFF,
    0x3FF0000000000000, 0xBFF0000000000000, 0x7FFFFFFFFFFFFFFF, 0xFFFFFFFFFFFFFFFF)]


def special_doubles(n, device, seed=0, out=None):
    """half the keys from SPECIAL_BITS, half normal doubles of either sign with magnitudes in [2^-10, 2^11)"""
    table = torch.tensor(SPECIAL_BITS, dtype=torch.int64, device=device)

    def f(h, i):
        mantissa = h & ((1 << 52) - 1)
        exponent = (1023 - 10 + ((h >> 52) & 31) % 21) << 52
        normal = mantissa | exponent | (h & INT64_MIN)
        pick = table[((h >> 58) & 63) % len(SPECIAL_BITS)]
        return torch.where((splitmix64(h) & 1) == 0, pick, normal)
    return _fill(n, device, seed, f, out)


def ragged_offsets(n, S, device, seed=0, long_segment=0):
    """offsets [S + 1] of S random segments over n elements; the first and the last are empty, and with long_segment
    > 0 one segment in the middle holds that many elements (the others share the rest, many of them empty)"""
    assert S >= 3 and 0 <= long_segment <= n
    rest = n - long_segment
    cuts = torch.sort(((splitmix64(torch.arange(S - 1, dtype=torch.int64, device=device) + (seed << 40)) >> 1)
                       % (rest + 1)))[0]
    cuts[0], cuts[-1] = 0, rest
    cuts[(S - 1) // 2:] += long_segment
    zero = torch.zeros(1, dtype=torch.int64, device=device)
    return torch.cat([zero, cuts, zero + n])
