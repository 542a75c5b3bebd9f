"""Host-side index arithmetic of the distributed sort, as plain integer/numpy functions.

These restate, for the host (planning, reporting, tests), what the kernels do on the device:
the block distribution of DistributedArray (mpi/mpi_lsbsort.cpp:109-120,144-149), the split of a
digit into sub-digits, the digit-major / rank-minor exclusive scan (:350,:385-414) and the
send-count matrix (:553-554).  Nothing here is on the sort's data path.
"""
import numpy as np


def div_ceil(a, b):
    return (a + b - 1) // b


def per_rank(n, ranks):
    """numElementsPerRank: ceil(n / ranks) (:144)"""
    return max(div_ceil(n, ranks), 1)


def elements_here(n, ranks, r):
    """numElementsHere with the reference's clamping (:145-149)"""
    per = per_rank(n, ranks)
    return max(min(per, n - per * r), 0)


def local_to_global(per, rank, loc):
    return rank * per + loc  # localIdxToGlobalIdx (:109-111)


def global_to_local(per, glb):
    rank = glb // per  # globalIdxToLocalIdx (:113-120)
    return rank, glb - rank * per


def num_passes(radix_bits, key_bits=64):
    """N_DIGITS (:22), ceil as chpl/arkouda-radix-sort.chpl:78-79; key_bits = 32 / 16 for a narrow key type"""
    return div_ceil(key_bits, radix_bits)


def plan_pass(radix_bits, digit, one_pass=False, key_bits=64):
    """(shift, bits, lo_bits, hi_bits) of reference pass `digit`: a digit wider than 8 bits is sorted as a
    stable low-sub-digit step followed by a stable high-sub-digit step, split evenly (fewer bins per step =
    longer runs per bin); LSB_FLAG_ONE_PASS sorts it by its low byte (K1) and then by the rest (K2).  The last digit
    is clamped to the key's width: key_bits = 32 / 16 for a narrow key type, whose order key fills the low key_bits
    bits of the key word (plan_pass in csrc/lsbsort.cu)"""
    shift = radix_bits * digit
    bits = min(radix_bits, key_bits - shift)
    lo = 0 if bits <= 8 else (8 if one_pass else bits // 2)
    return shift, bits, lo, bits - lo


def subpasses(radix_bits):
    out = []
    for d in range(num_passes(radix_bits)):
        shift, _, lo, hi = plan_pass(radix_bits, d)
        if lo:
            out.append((shift, lo))
        out.append((shift + lo, hi))
    return out


def global_starts(counts):
    """counts[rank][digit] -> starts[digit][rank]: exclusive scan in digit-major, rank-minor
    order, i.e. GlobalStarts[digit * R + rank] (:350,:407-413)"""
    counts = np.asarray(counts, dtype=np.int64)
    flat = counts.T.reshape(-1)
    starts = np.cumsum(flat) - flat
    return starts.reshape(counts.shape[1], counts.shape[0])


def send_counts(counts, per):
    """sendcounts[src][dst]: elements rank src sends to rank dst (:553-554), from counts alone"""
    counts = np.asarray(counts, dtype=np.int64)
    R = counts.shape[0]
    starts = global_starts(counts)
    out = np.zeros((R, R), dtype=np.int64)
    for r in range(R):
        b = starts[:, r]
        e = b + counts[r]
        for dst in range(R):
            lo, hi = dst * per, (dst + 1) * per
            out[r, dst] = np.clip(np.minimum(e, hi) - np.maximum(b, lo), 0, None).sum()
    return out


def remote_fraction(sent_row, me):
    """share of a shard's elements that leave the GPU in a pass (NVLink term of the roofline)"""
    total = int(sum(sent_row))
    return 0.0 if total == 0 else 1.0 - int(sent_row[me]) / total


def pass_roofline_ms(m, f_remote, hbm_gbs, nvlink_gbs):
    """SURVEY 8(d): t_pass >= max(m*32 B / BW_hbm, m*16 B*f_remote / BW_nvlink)"""
    return max(m * 32 / (hbm_gbs * 1e9), m * 16 * f_remote / (nvlink_gbs * 1e9)) * 1e3


def part_boundaries(per, V, ramp=1.3):
    """first local index of each of the V parts a shard of `per` slots is cut into for the pipelined multi-GPU
    pass (the same cut on every GPU), plus `per` at the end: equal parts for small shards, otherwise part sizes
    grow by `ramp` up to the middle of the shard and shrink again (lsb_create in csrc/lsbsort.cu)"""
    use_ramp = per >= V * 4096 and ramp > 1.0
    w = [ramp ** min(q, V - 1 - q) if use_ramp else 1.0 for q in range(V)]
    total, acc, out = sum(w), 0.0, [0]
    uniform = max(div_ceil(per, V), 1)
    for q in range(V):
        acc += w[q]
        e = int(per * (acc / total)) // 32 * 32 if use_ramp else (q + 1) * uniform
        if q == V - 1 or e > per:
            e = per
        out.append(max(e, out[-1]))
    return out


def bit_width(x):
    return int(x).bit_length() if x > 0 else 0


def segsort_layout(count, num_segments, radix_bits):
    """bit layout of a segmented sort (segsort_layout in csrc/lsb_segments.cuh): (idxbits, segbits, segw, passes, fits).
    The packed record carries the input index in idxbits = max(1, bits(count - 1)) bits below the segment id; after the
    key passes the key word becomes seg | idx << segw, segw = the segment id's segbits = bits(num_segments - 1) rounded
    up to whole digits, and the segment id is sorted by passes = segw / radix_bits more passes.  fits: both fields share
    one 64-bit word (all zero and False for num_segments < 1)."""
    if count < 0 or num_segments < 1 or not 1 <= radix_bits <= 16:
        return 0, 0, 0, 0, False
    idxbits = max(1, bit_width(count - 1))
    segbits = bit_width(num_segments - 1)
    passes = div_ceil(segbits, radix_bits)
    segw = passes * radix_bits
    return idxbits, segbits, segw, passes, segw + idxbits <= 64



def lexsort_rounds(widths, radix_bits):
    """rounds of a sort by key columns of widths 64 / 32 / 16 bits, least significant first (lexsort_rounds in
    csrc/lsb_lexsort.cuh): [(first, ncols, bits, passes)].  From column 0 on, the next column joins the current round while
    the round's summed width stays <= 64 and it holds fewer than 4 columns; bits is that sum, passes = ceil(bits / radix).
    Column first + c sits at the summed widths of the round's columns below it.  [] for no columns, a radix outside
    1..16 or another width."""
    if not widths or not 1 <= radix_bits <= 16 or any(w not in (16, 32, 64) for w in widths):
        return []
    rounds = []
    for c, w in enumerate(widths):
        if not rounds or rounds[-1][2] + w > 64 or rounds[-1][1] == 4:
            rounds.append([c, 0, 0])
        rounds[-1][1] += 1
        rounds[-1][2] += w
    return [(first, n, bits, div_ceil(bits, radix_bits)) for first, n, bits in rounds]

# ---- the one-pass kernel's work order (csrc/lsb_onepass.cuh), restated for tests ---------------------------------
def onepass_ticket(t, nsuper, t1, lead, tiles_last=None):
    """ticket t of the one-pass kernel -> ("K1", supertile, tile) | ("K2", supertile, segment) | None (no such item).
    A step is t1 K1 tickets (tile of supertile `step`) followed by 256 K2 tickets (segment of supertile `step - lead`)."""
    period = t1 + 256
    step, r = divmod(t, period)
    if step >= nsuper + lead:
        return None
    if r < t1:
        tiles = t1 if (tiles_last is None or step != nsuper - 1) else tiles_last
        return ("K1", step, r) if step < nsuper and r < tiles else None
    return ("K2", step - lead, r - t1) if step >= lead else None


def onepass_dependencies(item, nx, t1, tiles_last, nsuper):
    """the items a work item waits for: K1(s, .) overwrites scratch slot s % nx, so every segment of supertile s - nx
    must have gathered its pieces; K2(s, lo) needs every tile of supertile s in the scratch and the frontier of
    segment lo advanced past supertile s - 1"""
    kind, s, idx = item
    if kind == "K1":
        return [("K2", s - nx, lo) for lo in range(256)] if s >= nx else []
    tiles = tiles_last if s == nsuper - 1 else t1
    deps = [("K1", s, t) for t in range(tiles)]
    if s > 0:
        deps.append(("K2", s - 1, idx))
    return deps


# ---- the bucket plan of a one-GPU sort of 64-bit keys (plan_bucket / bucket_accepts in csrc/lsbsort.cu) -------------
def bucket_bytes(here, forced=0):
    """scatter steps on the top bytes before the bucket pass: the least k >= 2 with here <= 128 * 256^k (buckets of at
    most 128 records on average), or `forced` (tune key bk_bytes)"""
    if forced:
        return forced
    k = 2
    while k < 7 and here > 128 * 256 ** k:
        k += 1
    return k


def bucket_plan(byte_counts, here, radix_bits=16, no_skip=False, mode=0, forced=0):
    """k when a whole lsb_sort-type call of 64-bit keys on one GPU in the two-step shape takes the bucket plan (k stable
    steps on the top bytes, then the bucket pass), 0 when it runs the 8 byte steps.  byte_counts[s][b]: records whose
    order key has byte s equal to b.  mode: tune key bk_mode (0 auto, 1 never, 2 whenever the shape allows)."""
    if mode == 1 or radix_bits not in (8, 16) or here < 1 or (mode != 2 and here < 1 << 20):
        return 0
    k = bucket_bytes(here, forced)
    c = np.asarray(byte_counts, dtype=np.int64)
    if not no_skip and (c == here).any():
        return 0  # a constant byte: the byte steps skip it
    if mode != 2 and (c[8 - k:] * 128 > here).any():
        return 0  # a top byte with a bin over twice its share
    return k


def byte_counts(order_keys):
    """[8][256] counts of every byte of the order keys"""
    k = np.asarray(order_keys, dtype=np.uint64)
    return np.stack([np.bincount(((k >> np.uint64(8 * s)) & np.uint64(255)).astype(np.int64), minlength=256)
                     for s in range(8)])


def sort_stats(k, overflow=False, skipped=0):
    """(subpasses, partition_launches, kernel_launches) of a whole one-GPU sort in the two-step shape with one count
    launch over 8 byte steps: the bucket plan with k (0 = the byte steps, `skipped` of them skipped), and whether the
    bucket pass overflowed into the 8 byte steps"""
    if not k:
        steps = 8 - skipped
        return steps, steps, 2 + steps
    if overflow:
        return k + 8, k + 9, 2 + k + 1 + 8
    return 8, k + 1, 2 + k + 1
