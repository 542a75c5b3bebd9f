// lsb_unique.cuh -- the distinct keys or rows of K key columns (lsb_unique_device): the groups of equal elements, each
// group's first input position, every element's group and every group's size.  Columns and rounds are lexsort's
// (lsb_lexsort.cuh); two elements are equal when every column's order key is.
//
// Sorted mode runs lexsort's packs and passes first, so that buf[cur][p] = {the last round's word, input index} of the
// p-th record in lexsort order; consecutive mode reads the columns in input order and sorts nothing.  Position p >= 1
// starts a group (is a head) when its words differ from those of position p - 1 in some round:
//
//   unique_flag_kernel<SORTED, N>   diff[p-1] (|)= word_r(p) != word_r(p-1), one launch per round but the last
//                                   (sorted: 16 read + 2 random W_c / 8 per column, only lane 0 of a warp reads its
//                                   neighbour's; consecutive: Σ W_c / 8 read; 1 written, 1 read by every later launch)
//   unique_tile_kernel<0, N>        totals[t] = heads in tile t                    (16 read sorted, Σ W_c / 8 consecutive;
//                                                                                  + 1 with diff)
//   global_scan_kernel (G = 1)      bases = exclusive scan of totals               (16 per tile)
//   unique_tile_kernel<1, N>        heads again, r = group of p = bases[t] + heads in [tile start, p] - 1:
//                                   index_out[r] = input index of a head; ends[r-1] = p for a head, r >= 1;
//                                   inverse_out[input index of p] = r               (the reads of phase 0, 8 written per head
//                                                                                  for each of index and ends, 8 per element
//                                                                                  for inverse: random in sorted mode)
//   unique_counts_kernel            counts[r] = ends[r] - ends[r-1], ends[-1] = 0, ends[U-1] = count   (16 + 8 per group)
//
// N = 0 reads the last round's word from the sorted records, N = 1..4 folds the last round's columns (consecutive mode).
// The head flags of the last round are never stored: both tile phases compute them again, from the same loads.
#pragma once
#include "lsb_lexsort.cuh"

namespace lsb {

constexpr int UNIQUE_THREADS = 256;
constexpr int UNIQUE_ITEMS = 8;
constexpr int UNIQUE_TILE = UNIQUE_THREADS * UNIQUE_ITEMS;

// The scratch of a call of `count` >= 1 elements: ends int64[count - 1], totals u64[T], bases int64[T] and diff
// uint8[count - 1], T = ceil(count / UNIQUE_TILE), in this order.  9 (count - 1) + 16 T <= 16 count for every count >= 1,
// so they fit the shard buffer the passes do not hold (16 bytes per element).
struct UniqueScratch {
  int64_t* ends;
  unsigned long long* totals;
  int64_t* bases;
  uint8_t* diff;
  int64_t tiles;
};

__host__ __device__ inline UniqueScratch unique_scratch(void* base, int64_t count) {
  UniqueScratch s;
  s.tiles = (count + UNIQUE_TILE - 1) / UNIQUE_TILE;
  s.ends = (int64_t*)base;
  s.totals = (unsigned long long*)(s.ends + (count - 1));
  s.bases = (int64_t*)(s.totals + s.tiles);
  s.diff = (uint8_t*)(s.bases + s.tiles);
  return s;
}

#ifdef __CUDACC__

// the round word of element j: the OR of its NCOLS columns' order keys at their shifts (lexsort_pack_kernel's word)
template <int NCOLS>
__device__ __forceinline__ uint64_t unique_word(const LexsortColumn* col, int64_t j) {
  uint64_t raw[NCOLS], w = 0;
#pragma unroll
  for (int c = 0; c < NCOLS; c++) raw[c] = NCOLS == 1 ? lexsort_load(col[c], j) : lexsort_load_narrow(col[c], j);
#pragma unroll
  for (int c = 0; c < NCOLS; c++) w |= lexsort_order(col[c], raw[c]);
  return w;
}

struct UniqueFlagArgs {
  LexsortColumn col[LEXSORT_ROUND_COLUMNS];  // the round's NCOLS columns
  const Elt* rec;  // SORTED: the sorted records, whose val word is the input index of position p
  uint8_t* diff;   // [count - 1]
  int64_t count;
  int first;       // the first round flagged: diff is written, not ORed into
};

// One earlier round's flags.  A warp covers 32 consecutive positions, so position p - 1's word comes from the lane below;
// lane 0 computes it again.  All IO_U positions of a thread have their loads in flight before the first fold.
template <bool SORTED, int NCOLS>
__global__ void __launch_bounds__(IO_THREADS) unique_flag_kernel(const UniqueFlagArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  for (int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; i - lane < a.count; i += IO_U * stride) {
    int64_t idx[IO_U], prev_idx[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t p = i + u * stride;
      idx[u] = prev_idx[u] = 0;
      if (p < a.count) idx[u] = SORTED ? (int64_t)ld_stream(a.rec + p).val : p;
      if (lane == 0 && p > 0 && p < a.count) prev_idx[u] = SORTED ? (int64_t)ld_stream(a.rec + p - 1).val : p - 1;
    }
    uint64_t w[IO_U], prev[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      w[u] = prev[u] = 0;
      if (i + u * stride < a.count) w[u] = unique_word<NCOLS>(a.col, idx[u]);
      if (lane == 0 && i + u * stride > 0 && i + u * stride < a.count) prev[u] = unique_word<NCOLS>(a.col, prev_idx[u]);
    }
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      const int64_t p = i + u * stride;
      const uint64_t below = __shfl_up_sync(0xffffffffu, w[u], 1);
      if (lane) prev[u] = below;
      if (p > 0 && p < a.count) {
        const uint8_t d = w[u] != prev[u];
        a.diff[p - 1] = a.first ? d : (uint8_t)(a.diff[p - 1] | d);
      }
    }
  }
}

struct UniqueTileArgs {
  const Elt* rec;                            // NCOLS = 0: the sorted records {last round's word, input index}
  LexsortColumn col[LEXSORT_ROUND_COLUMNS];  // NCOLS >= 1: the last round's columns, read at p
  const uint8_t* diff;                       // the earlier rounds' flags, or nullptr for a single round
  int64_t count;
  unsigned long long* totals;                // [tiles]: written by phase 0
  const int64_t* bases;                      // [tiles]: read by phase 1
  int64_t* index_out;                        // phase 1, each may be nullptr
  int64_t* inverse_out;
  int64_t* ends;
  int64_t* num_unique;                       // phase 1: U, written by the last tile
};

// Tile blockIdx.x: item k of thread t is position tile0 + k * UNIQUE_THREADS + t.  PHASE 0 counts the tile's heads,
// PHASE 1 numbers them and writes the outputs.
template <int PHASE, int NCOLS>
__global__ void __launch_bounds__(UNIQUE_THREADS) unique_tile_kernel(const UniqueTileArgs a) {
  constexpr int WARPS = UNIQUE_THREADS / 32;
  __shared__ uint32_t s_cnt[UNIQUE_ITEMS * WARPS];  // heads of item k in warp w at [k * WARPS + w], then their scan
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t tile0 = (int64_t)blockIdx.x * UNIQUE_TILE + threadIdx.x;
  uint64_t w[UNIQUE_ITEMS], prev[UNIQUE_ITEMS];
  int64_t idx[UNIQUE_ITEMS];
#pragma unroll
  for (int k = 0; k < UNIQUE_ITEMS; k++) {
    const int64_t p = tile0 + k * UNIQUE_THREADS;
    w[k] = prev[k] = 0;
    idx[k] = p;
    if (p < a.count) {
      if (NCOLS == 0) {
        const Elt e = ld_stream(a.rec + p);
        w[k] = e.key;
        idx[k] = (int64_t)e.val;
      } else {
        w[k] = unique_word<NCOLS ? NCOLS : 1>(a.col, p);
      }
    }
    if (lane == 0 && p > 0 && p < a.count)
      prev[k] = NCOLS == 0 ? ld_stream_key(a.rec + p - 1) : unique_word<NCOLS ? NCOLS : 1>(a.col, p - 1);
  }
  uint32_t heads = 0;
#pragma unroll
  for (int k = 0; k < UNIQUE_ITEMS; k++) {
    const int64_t p = tile0 + k * UNIQUE_THREADS;
    const uint64_t below = __shfl_up_sync(0xffffffffu, w[k], 1);
    if (lane) prev[k] = below;
    const bool head = p < a.count && (p == 0 || w[k] != prev[k] || (a.diff && a.diff[p - 1]));
    heads |= (uint32_t)head << k;
  }
  uint32_t ballot[UNIQUE_ITEMS];
#pragma unroll
  for (int k = 0; k < UNIQUE_ITEMS; k++) {
    ballot[k] = __ballot_sync(0xffffffffu, (heads >> k) & 1);
    if (lane == 0) s_cnt[k * WARPS + warp] = __popc(ballot[k]);
  }
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the UNIQUE_ITEMS * WARPS = 64 counts in position order: 2 per lane
    static_assert(UNIQUE_ITEMS * WARPS == 64, "one warp scans two counts per lane");
    const uint32_t c0 = s_cnt[2 * lane], c1 = s_cnt[2 * lane + 1];
    const uint32_t incl = (uint32_t)warp_incl_scan(c0 + c1);
    if (PHASE == 0) {
      if (lane == 31) a.totals[blockIdx.x] = incl;
    } else {
      s_cnt[2 * lane] = incl - c0 - c1;
      s_cnt[2 * lane + 1] = incl - c1;
      if (lane == 31 && blockIdx.x == gridDim.x - 1) *a.num_unique = a.bases[blockIdx.x] + incl;
    }
  }
  if (PHASE == 0) return;
  __syncthreads();
  const int64_t base = a.bases[blockIdx.x];
#pragma unroll
  for (int k = 0; k < UNIQUE_ITEMS; k++) {
    const int64_t p = tile0 + k * UNIQUE_THREADS;
    if (p >= a.count) break;
    // the group of p: heads before the tile, plus heads up to and including p, less one (p = 0 is always a head)
    const int64_t r = base + s_cnt[k * WARPS + warp] + __popc(ballot[k] & (lanemask_lt() | (1u << lane))) - 1;
    if ((heads >> k) & 1) {
      if (a.index_out) a.index_out[r] = idx[k];
      if (a.ends && r > 0) a.ends[r - 1] = p;
    }
    if (a.inverse_out) a.inverse_out[idx[k]] = r;
  }
}

struct UniqueCountsArgs {
  const int64_t* ends;        // [U - 1]
  const int64_t* num_unique;  // U, on the device
  int64_t* counts;
  int64_t count;
};

__global__ void __launch_bounds__(IO_THREADS) unique_counts_kernel(const UniqueCountsArgs a) {
  const int64_t u = *a.num_unique, stride = (int64_t)gridDim.x * IO_THREADS;
  for (int64_t r = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x; r < u; r += stride)
    a.counts[r] = (r + 1 < u ? a.ends[r] : a.count) - (r ? a.ends[r - 1] : 0);
}

#endif  // __CUDACC__

}  // namespace lsb
