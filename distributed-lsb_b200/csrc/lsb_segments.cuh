// lsb_segments.cuh -- the streams around a segmented sort (lsb_sort_segments_device): many independent groups, segment s
// being the input positions [offsets[s], offsets[s+1]), sorted at once as ONE stable LSD sort by (s, order_key(key)).
//
// Named segsort_* so as not to be confused with the partition kernel's seg_start / seg_tiles or the one-pass kernel's
// K2 segments.  The sort between them is lsb_sort's, unchanged:
//
//   segsort_check_kernel   offsets[0] == 0, offsets[S] == count, non-decreasing              -> one flag
//   segsort_pack_kernel    dst[i] = {key_word(key[i]), i | seg(i) << idxbits}                 (24 B/element + offsets)
//   ... the key passes of lsb_sort (every pass shape and key order) ...
//   segsort_retag_kernel   {key, idx | seg << idxbits} -> {seg | idx << segw, key}, in place  (32 B/element)
//   ... segw / radix_bits passes on the low digits of the new key word, uint64 ascending ...
//   segsort_unpack_kernel  keys_out[i] = key of the val word; vals_out[i] = vals_in[idx] | idx - offsets[seg] | idx
//
// The key word is the 8-byte key itself, or for a narrow key type (lsb_sort_segments_device_typed) narrow_key_word:
// the pack templated on the LSB_KEY_* type reads W-bit keys, the unpack templated on KBYTES writes the word's high half.
// The key passes then cover the low W bits only; the retag and the segment passes move the whole word unchanged.
//
// The key passes leave equal (key) records in index order, so after the stable segment passes every segment holds its
// records sorted by key and ties in input order: the stable sort by (seg, key).  A single segment (segbits == 0) needs
// neither the segment id nor the retag: the call is then lsb_sort_device's pack_kernel / unpack_kernel around the sort.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#include "lsb_io.cuh"
#endif

namespace lsb {

// Bit layout of a segmented sort of `count` elements in `num_segments` segments at radix `radix_bits`, shared by the
// library and the tests (distributed-lsb_b200/hostlogic.py restates it):
//   idxbits = bit width of count - 1, at least 1       (the input index, low bits of the packed val word)
//   segbits = bit width of num_segments - 1            (the segment id; 0: one segment, no segment passes)
//   segw    = radix_bits * ceil(segbits / radix_bits)  (the segment id's field after the retag: whole digits)
//   passes  = segw / radix_bits                        (segment passes after the key passes)
//   fits    = segw + idxbits <= 64                     (both fields in one key word; false also for num_segments < 1)
struct SegsortLayout {
  int idxbits, segbits, segw, passes;
  bool fits;
};

__host__ __device__ inline int segsort_bit_width(int64_t x) {
  int w = 0;
  while (w < 63 && (x >> w) > 0) w++;
  return w;
}

__host__ __device__ inline SegsortLayout segsort_layout(int64_t count, int64_t num_segments, int radix_bits) {
  SegsortLayout l = {0, 0, 0, 0, false};
  if (count < 0 || num_segments < 1 || radix_bits < 1 || radix_bits > 16) return l;
  const int w = segsort_bit_width(count - 1);
  l.idxbits = w > 1 ? w : 1;
  l.segbits = segsort_bit_width(num_segments - 1);
  l.passes = (l.segbits + radix_bits - 1) / radix_bits;
  l.segw = l.passes * radix_bits;
  l.fits = l.segw + l.idxbits <= 64;
  return l;
}

#ifdef __CUDACC__

struct SegsortCheckArgs {
  const int64_t* offsets;  // [nseg + 1]
  int64_t nseg;
  int64_t count;
  int* bad;                // set to 1 by any failed check (zeroed by the caller)
};

__global__ void __launch_bounds__(IO_THREADS) segsort_check_kernel(const SegsortCheckArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  bool bad = false;
  for (int64_t s0 = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; s0 < a.nseg; s0 += IO_U * stride) {
    int64_t lo[IO_U], hi[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t s = s0 + u * stride;
      lo[u] = s < a.nseg ? (int64_t)ld_stream_u64((const uint64_t*)a.offsets + s) : 0;
      hi[u] = s < a.nseg ? (int64_t)ld_stream_u64((const uint64_t*)a.offsets + s + 1) : 0;
    }
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t s = s0 + u * stride;
      bad = bad || lo[u] > hi[u] || (s == 0 && lo[u] != 0) || (s == a.nseg - 1 && hi[u] != a.count);
    }
  }
  if (bad) *a.bad = 1;
}

// largest s in [s, s + len) with off[min(s', nseg)] <= t, given off[s] <= t: the segment of input position t when the
// range holds it.  The steps depend on `len` alone, so a warp with one len runs them in lockstep.  Positions past the
// range are never taken (their offsets exceed t) and the read is clamped to off[nseg] = count > t.
__device__ __forceinline__ void segsort_search(const int64_t* off, int64_t nseg, int64_t len, const int64_t (&t)[IO_U],
                                               int64_t (&s)[IO_U]) {
  while (len > 1) {
    const int64_t half = len >> 1;
    int64_t p[IO_U], o[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) p[u] = min(s[u] + half, nseg);
#pragma unroll
    for (int u = 0; u < IO_U; u++) o[u] = __ldg(off + p[u]);
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (o[u] <= t[u]) s[u] = p[u];
    len -= half;
  }
}

struct SegsortPackArgs {
  const void* keys;
  const int64_t* offsets;  // [nseg + 1], checked by segsort_check_kernel
  Elt* dst;                // shard buf[0]
  int64_t count;
  int64_t nseg;
  int idxbits;
  uint32_t flags;          // narrow KT: the key order (DESCENDING) applied to the key word
};

// Warp w of a CTA handles the 32 consecutive elements base + lane of each of its IO_U groups.  Two lanes find the
// segments of the group's first and last element in all of offsets (one lockstep search); every lane then searches only
// between those two, which for segments of >= 32 elements is zero or one step.
template <int KT>
__global__ void __launch_bounds__(IO_THREADS) segsort_pack_kernel(const SegsortPackArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  const int64_t last = a.count - 1;
  for (int64_t base = (int64_t)blockIdx.x * IO_THREADS + (threadIdx.x & ~31); base < a.count; base += IO_U * stride) {
    uint64_t k[IO_U];
    int64_t t[IO_U], s[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t i = base + u * stride + lane;
      k[u] = i < a.count ? ld_key_word<KT>(a.keys, i, a.flags) : 0;
      t[u] = min(base + u * stride + ((lane & 1) ? 31 : 0), last);  // even lanes: first element, odd lanes: last
      s[u] = 0;
    }
    segsort_search(a.offsets, a.nseg, a.nseg, t, s);
    int64_t width = 1;
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t first_seg = __shfl_sync(0xffffffffu, s[u], 0), last_seg = __shfl_sync(0xffffffffu, s[u], 1);
      width = max(width, last_seg - first_seg + 1);
      s[u] = first_seg;
      t[u] = min(base + u * stride + lane, last);
    }
    segsort_search(a.offsets, a.nseg, width, t, s);
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t i = base + u * stride + lane;
      if (i < a.count) st_elt(a.dst + i, Elt{k[u], (uint64_t)i | ((uint64_t)s[u] << a.idxbits)});
    }
  }
}

struct SegsortRetagArgs {
  Elt* buf;  // shard buf[cur] after the key passes, rewritten in place
  int64_t count;
  int idxbits;
  int segw;
};

__global__ void __launch_bounds__(IO_THREADS) segsort_retag_kernel(const SegsortRetagArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  const uint64_t idx_mask = (1ULL << a.idxbits) - 1;
  for (int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; i < a.count; i += IO_U * stride) {
    Elt e[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count) e[u] = ld_stream(a.buf + i + u * stride);
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count)
        st_elt(a.buf + i + u * stride, Elt{(e[u].val >> a.idxbits) | ((e[u].val & idx_mask) << a.segw), e[u].key});
  }
}

// what vals_out receives
enum SegsortVals { SEGSORT_VALS_NONE = 0, SEGSORT_VALS_GATHER = 1, SEGSORT_VALS_LOCAL = 2, SEGSORT_VALS_GLOBAL = 3 };

struct SegsortUnpackArgs {
  const Elt* src;          // shard buf[cur] after the segment passes: {seg | idx << segw, key}
  void* keys;              // KEYS only
  uint64_t* vals;          // VALS != NONE only
  const uint64_t* vals_in; // GATHER
  const int64_t* offsets;  // LOCAL
  int64_t count;
  int segw;
};

template <int KBYTES, bool KEYS, int VALS>
__global__ void __launch_bounds__(IO_THREADS) segsort_unpack_kernel(const SegsortUnpackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  const uint64_t seg_mask = (1ULL << a.segw) - 1;
  for (int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; i < a.count; i += IO_U * stride) {
    Elt e[IO_U];
    uint64_t v[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count) e[u] = ld_stream(a.src + i + u * stride);
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      if (i + u * stride >= a.count) continue;
      const uint64_t idx = e[u].key >> a.segw;
      if (VALS == SEGSORT_VALS_GATHER) v[u] = __ldg(a.vals_in + idx);
      else if (VALS == SEGSORT_VALS_LOCAL) v[u] = idx - (uint64_t)__ldg(a.offsets + (e[u].key & seg_mask));
      else v[u] = idx;
    }
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      if (i + u * stride >= a.count) continue;
      if (KEYS) st_key<KBYTES>(a.keys, i + u * stride, e[u].val);
      if (VALS != SEGSORT_VALS_NONE) a.vals[i + u * stride] = v[u];
    }
  }
}

#endif  // __CUDACC__

}  // namespace lsb
