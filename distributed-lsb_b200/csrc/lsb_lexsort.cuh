// lsb_lexsort.cuh -- the streams around a sort by several key columns (lsb_lexsort_device): K columns of any key type,
// columns[0] the least significant and columns[K-1] the primary, as np.lexsort orders them.
//
// The columns are cut into rounds (lexsort_rounds): consecutive columns, least significant first, whose widths sum to
// at most 64 bits share one key word.  A round's word is the OR of its columns' order keys, each shifted above the
// round's less significant columns, so one run of stable passes on its `bits` low bits sorts by all of them at once.
// The rounds run least significant first; each is stable, so a later round keeps the order of the earlier ones for
// records equal in its own columns:
//
//   lexsort_pack_kernel<false, N>  buf[0][i] = {word_0(i), i}                                   (Σ W_c / 8 read, 16 written)
//   ... the passes of round 0 ...
//   lexsort_pack_kernel<true, N>   e = buf[cur][p]; buf[cur][p] = {word_r(e.val), e.val}      (16 + a random W_c / 8 per
//   ... the passes of round r ...                                                            column read, 16 written)
//   lexsort_unpack_kernel       vals_out[p] = vals_in[buf[cur][p].val]                       (16 + a random 8 read, 8 written)
//                               (without vals_in, unpack_kernel<8, false, true> writes the index itself)
//
// The val word always holds the input index.  order_c is order_key (8-byte column) or order_key_narrow (lsb_keyorder.cuh)
// under the column's own flags, so every pass reads its word as a uint64 ascending (the ORD = false kernels).
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#include <type_traits>

#include "lsb_io.cuh"
#endif

namespace lsb {

constexpr int LEXSORT_ROUND_COLUMNS = 4;  // 4 x 16 bits fill a key word

// Round r of a lexsort: columns [first, first + ncols) in one key word of `bits` bits (their summed widths), sorted by
// passes = ceil(bits / radix_bits) passes.  Column first + c sits at the summed widths of columns first .. first + c - 1.
struct LexsortRound {
  int first, ncols, bits, passes;
};

// The rounds of K columns of widths 64 / 32 / 16 at radix radix_bits (distributed-lsb_b200/hostlogic.py restates it):
// from columns[0] on, the next column joins the current round while the round's summed width stays at most 64 bits and
// it holds fewer than 4 columns.  Greedy packing of consecutive columns gives the fewest rounds.  Writes at most K
// rounds to `rounds` and returns their number; 0 for K < 1, a radix outside 1..16 or another width.
__host__ __device__ inline int lexsort_rounds(const int* widths, int K, int radix_bits, LexsortRound* rounds) {
  if (K < 1 || radix_bits < 1 || radix_bits > 16) return 0;
  int n = 0;
  for (int c = 0; c < K; c++) {
    const int w = widths[c];
    if (w != 64 && w != 32 && w != 16) return 0;
    if (n == 0 || rounds[n - 1].bits + w > 64 || rounds[n - 1].ncols == LEXSORT_ROUND_COLUMNS) rounds[n++] = {c, 0, 0, 0};
    rounds[n - 1].ncols++;
    rounds[n - 1].bits += w;
  }
  for (int r = 0; r < n; r++) rounds[r].passes = (rounds[r].bits + radix_bits - 1) / radix_bits;
  return n;
}

#ifdef __CUDACC__

struct LexsortColumn {
  const void* keys;   // count keys of key_type
  uint32_t key_type;  // LSB_KEY_CONTEXT (8-byte, ordered by flags) .. LSB_KEY_BF16
  uint32_t flags;     // LSB_FLAG_DESCENDING, and KEY_I64 / KEY_F64 for an 8-byte column
  int shift;          // of its order key in the round's word
};

struct LexsortPackArgs {
  LexsortColumn col[LEXSORT_ROUND_COLUMNS];  // the round's NCOLS columns
  Elt* buf;  // GATHER = false: shard buf[0], written; GATHER = true: shard buf[cur], rewritten in place
  int64_t count;
};

// The raw bits of key j of a column and their order key at the column's shift.  A round of one column may hold any
// width; a round of NCOLS >= 2 columns holds narrow ones only (64 + 16 > 64), whose raw bits fit 32 bits.  The type is
// uniform over the grid, so the branches never diverge.
__device__ __forceinline__ uint32_t lexsort_load_narrow(const LexsortColumn& c, int64_t j) {
  return key_type_bits(c.key_type) == 32 ? ld_stream_u32((const uint32_t*)c.keys + j) : ld_stream_u16((const uint16_t*)c.keys + j);
}

__device__ __forceinline__ uint64_t lexsort_load(const LexsortColumn& c, int64_t j) {
  if (c.key_type == LSB_KEY_CONTEXT) return ld_stream_u64((const uint64_t*)c.keys + j);
  return lexsort_load_narrow(c, j);
}

__device__ __forceinline__ uint64_t lexsort_order(const LexsortColumn& c, uint64_t k) {
  const uint64_t o = c.key_type == LSB_KEY_CONTEXT ? order_key(k, c.flags) : order_key_narrow((uint32_t)k, c.key_type, c.flags);
  return o << c.shift;
}

// IO_U elements of a thread in flight: (GATHER) their records, then the keys of all NCOLS columns, then the stores.
// The round's column count is a template parameter so that no column's loads wait behind a check or a fold of the one
// before.
template <bool GATHER, int NCOLS>
__global__ void __launch_bounds__(IO_THREADS, IO_CTAS_PER_SM) lexsort_pack_kernel(const LexsortPackArgs a) {
  using Raw = typename std::conditional<NCOLS == 1, uint64_t, uint32_t>::type;
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  for (int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; i < a.count; i += IO_U * stride) {
    uint64_t idx[IO_U];
    Raw k[NCOLS][IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      idx[u] = 0;
      if (i + u * stride < a.count) idx[u] = GATHER ? ld_stream(a.buf + i + u * stride).val : (uint64_t)(i + u * stride);
    }
#pragma unroll
    for (int c = 0; c < NCOLS; c++)
#pragma unroll
      for (int u = 0; u < IO_U; u++)
        if (i + u * stride < a.count)
          k[c][u] = NCOLS == 1 ? (Raw)lexsort_load(a.col[c], (int64_t)idx[u]) : (Raw)lexsort_load_narrow(a.col[c], (int64_t)idx[u]);
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      if (i + u * stride >= a.count) continue;
      uint64_t word = 0;
#pragma unroll
      for (int c = 0; c < NCOLS; c++) word |= lexsort_order(a.col[c], k[c][u]);
      st_elt(a.buf + i + u * stride, Elt{word, idx[u]});
    }
  }
}

struct LexsortUnpackArgs {
  const Elt* src;           // shard buf[cur] after the last round
  const uint64_t* vals_in;  // gathered by the input index in the val word
  uint64_t* vals;
  int64_t count;
};

__global__ void __launch_bounds__(IO_THREADS) lexsort_unpack_kernel(const LexsortUnpackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  for (int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; i < a.count; i += IO_U * stride) {
    uint64_t idx[IO_U], v[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count) idx[u] = ld_stream(a.src + i + u * stride).val;
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count) v[u] = __ldg(a.vals_in + idx[u]);
#pragma unroll
    for (int u = 0; u < IO_U; u++)
      if (i + u * stride < a.count) a.vals[i + u * stride] = v[u];
  }
}

#endif  // __CUDACC__

}  // namespace lsb
