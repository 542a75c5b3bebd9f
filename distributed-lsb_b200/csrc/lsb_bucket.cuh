// lsb_bucket.cuh -- the bucket pass of a one-GPU sort of 64-bit keys (sm_100a).
//
// Input: records stably sorted by top = order_key(key) >> top_shift (the k scatter steps on the top k bytes).  Every
// run of equal top (a bucket) holds 2^(64 - 8k) possible low values and, by the plan's choice of k, about 64 records
// on average (at most 128).  Output: the same records stably sorted by order_key(key), at the same global positions
// in the other buffer, so reads and stores are contiguous streams and the pass costs one trip through HBM.
//
// A CTA owns the buckets whose first record lies in its tile [t0, t0 + BK_TILE).  It loads [t0 - 1, t0 + BK_TILE +
// BK_C) clipped to [0, n) with one bulk copy: record t0 - 1 decides whether t0 starts a bucket, the halo of BK_C
// records finishes the last owned bucket.  The CTA marks bucket boundaries in a bit mask, then warp w takes the
// buckets starting in its BK_SEG records and packs consecutive whole buckets into chunks of at most BK_C records.  A
// chunk is sorted in the warp's registers (a bitonic network of 64, 128 or 256 keys: 2, 4 or 8 per lane) by the key
//   ordinal << ord_shift | low << 8 | pos
// ordinal = index of the record's bucket in the chunk (monotone in top, so it stands for the top bits), low = the low
// 64 - 8k bits of order_key, pos = index in the chunk (equal keys keep their order).  For k >= 2 and BK_C <= 256 that
// fills at most 64 bits, and a chunk with padding has fewer than 256 records, so its ordinals stay below 255 and the
// padding key ~0 sorts after every record.  Lane-major stores then write rank r of the chunk to chunk start + r.
//
// A bucket longer than BK_C is streamed through its warp from global memory instead (bk_long_bucket): when its order
// keys are already in order -- all equal, as the NaNs of a float64 sort or a repeated key -- it is copied as it is.
// Otherwise it sets *overflow: the caller then sorts the kernel's input again with the byte steps (the input is a stable
// permutation of the original by the top bits, so a stable sort of it is the stable sort of the original), and whatever
// this launch stored is overwritten.
#pragma once
#include "lsb_kernels.cuh"

namespace lsb {

constexpr int BK_THREADS = 512;
constexpr int BK_WARPS = BK_THREADS / 32;
constexpr int BK_TILE = 4096;                  // records whose buckets one CTA owns
constexpr int BK_C = 256;                      // largest chunk (and bucket) one warp sorts: 8 keys per lane
constexpr int BK_SEG = BK_TILE / BK_WARPS;     // records of the tile whose buckets one warp owns
constexpr int BK_WIN = 1 + BK_TILE + BK_C;     // records a CTA loads
constexpr int BK_WORDS = (BK_WIN + 1 + 31) / 32;  // boundary bits of window positions 0..BK_WIN
// loaded window | per-warp chunk keys (u64, swizzled), later the chunk's rank -> position bytes | boundary bits
constexpr int BK_SMEM_KEYS = BK_WIN * 16;
constexpr int BK_SMEM_BITS = BK_SMEM_KEYS + BK_WARPS * BK_C * 8;
constexpr int BK_SMEM = BK_SMEM_BITS + BK_WORDS * 4;
static_assert(BK_SEG + BK_C <= 32 * 32 && BK_C == 256, "searches span at most 32 words; the network is 8 keys per lane");

struct BucketArgs {
  const Elt* src;
  Elt* dst;
  int64_t n;
  int top_shift;       // 64 - 8k
  int ord_shift;       // 72 - 8k
  uint64_t low_mask;   // (1 << (64 - 8k)) - 1
  unsigned* overflow;  // set to 1 when a bucket longer than BK_C is out of order (caller zeroes)
  uint32_t korder;
};

// chunk key slot of chunk index e: lane-major writes (e = r * 32 + lane) and register-major reads (e = lane * 8 + r)
// both touch 16 distinct 8-byte slots per half warp
__device__ __forceinline__ int bk_swz(int e) { return e ^ ((e >> 3) & 15); }

__device__ __forceinline__ bool bk_bit(const unsigned* bits, int i) { return (bits[i >> 5] >> (i & 31)) & 1u; }

// last set bit of bits[] in [lo, hi] (hi - lo < 32 * 31), or -1; warp-uniform arguments and result
__device__ __forceinline__ int bk_find_last(const unsigned* bits, int lo, int hi, int lane) {
  if (hi < lo) return -1;
  const int wd = (hi >> 5) - lane;
  unsigned w = 0;
  if (wd >= (lo >> 5)) {
    w = bits[wd];
    if (wd == (hi >> 5)) w &= 0xffffffffu >> (31 - (hi & 31));
    if (wd == (lo >> 5)) w &= 0xffffffffu << (lo & 31);
  }
  const unsigned any = __ballot_sync(0xffffffffu, w != 0);
  if (!any) return -1;
  const int src = __ffs(any) - 1;  // the lowest lane holds the highest word
  const unsigned sw = __shfl_sync(0xffffffffu, w, src);
  return ((hi >> 5) - src) * 32 + 31 - __clz(sw);
}

// first set bit of bits[] in [lo, hi] (hi - lo < 32 * 31), or -1
__device__ __forceinline__ int bk_find_first(const unsigned* bits, int lo, int hi, int lane) {
  if (hi < lo) return -1;
  const int wd = (lo >> 5) + lane;
  unsigned w = 0;
  if (wd <= (hi >> 5)) {
    w = bits[wd];
    if (wd == (hi >> 5)) w &= 0xffffffffu >> (31 - (hi & 31));
    if (wd == (lo >> 5)) w &= 0xffffffffu << (lo & 31);
  }
  const unsigned any = __ballot_sync(0xffffffffu, w != 0);
  if (!any) return -1;
  const int src = __ffs(any) - 1;
  const unsigned sw = __shfl_sync(0xffffffffu, w, src);
  return ((lo >> 5) + src) * 32 + __ffs(sw) - 1;
}

// ascending bitonic sort of 32 * R keys, key (lane * R + r) in k[r]
template <int R>
__device__ __forceinline__ void bk_bitonic(uint64_t (&k)[R], int lane) {
#pragma unroll
  for (int kk = 2; kk <= 32 * R; kk <<= 1) {
#pragma unroll
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= R) {  // partner in lane ^ (j / R), same register
        const int lj = j / R;
        const bool up = ((lane * R) & kk) == 0;
        const bool keep_max = up == ((lane & lj) != 0);
#pragma unroll
        for (int r = 0; r < R; r++) {
          const uint64_t o = __shfl_xor_sync(0xffffffffu, k[r], lj);
          k[r] = ((o < k[r]) != keep_max) ? o : k[r];
        }
      } else {  // partner in register r ^ j, same lane
#pragma unroll
        for (int r = 0; r < R; r++) {
          if (r & j) continue;
          const bool up = ((lane * R + r) & kk) == 0;
          const uint64_t a = k[r], b = k[r | j];
          const bool sw = up ? (b < a) : (a < b);
          k[r] = sw ? b : a;
          k[r | j] = sw ? a : b;
        }
      }
    }
  }
}

// the chunk [p, p + len) of window positions, len <= 32 * R, sorted by its chunk keys and stored to dst + w0 + p
template <int R, bool ORD>
__device__ __forceinline__ void bk_sort_chunk(const BucketArgs& a, const Elt* s_raw, const unsigned* bits, uint64_t* keys,
                                              int p, int len, int64_t w0, int lane) {
  // chunk keys, lane-major
  int ordinal = 0;
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int e = r * 32 + lane;
    const bool in = e < len;
    const bool start = in && e > 0 && bk_bit(bits, p + e);
    const unsigned b = __ballot_sync(0xffffffffu, start);
    uint64_t key = ~0ull;
    if (in) {
      const uint64_t ok = digit_key<ORD>(s_raw[p + e].key, a.korder);
      key = (uint64_t)(ordinal + __popc(b & (lanemask_lt() << 1 | 1u))) << a.ord_shift | (ok & a.low_mask) << 8 | (uint64_t)e;
    }
    ordinal += __popc(b);
    keys[bk_swz(e)] = key;
  }
  __syncwarp();
  uint64_t k[R];
#pragma unroll
  for (int r = 0; r < R; r++) k[r] = keys[bk_swz(lane * R + r)];
  __syncwarp();
  bk_bitonic<R>(k, lane);
  unsigned char* perm = reinterpret_cast<unsigned char*>(keys);  // chunk position of rank e: perm[e]
#pragma unroll
  for (int r = 0; r < R; r++) perm[lane * R + r] = (unsigned char)k[r];
  __syncwarp();
  Elt* out = a.dst + w0 + p;
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int e = r * 32 + lane;
    if (e < len) st_elt(out + e, s_raw[p + perm[e]]);
  }
  __syncwarp();
}

// A bucket of more than BK_C records starting at global index g0, streamed through the warp from global memory: when its
// order keys are already non-decreasing (equal keys: the NaNs of a float64 sort, a repeated key), its stable sort is the
// identity and it is copied to dst as it is.  Returns false when it is out of order (the caller reports an overflow).
template <bool ORD>
__device__ __noinline__ bool bk_long_bucket(const BucketArgs& a, int64_t g0, int lane) {
  const uint64_t top0 = digit_key<ORD>(a.src[g0].key, a.korder) >> a.top_shift;
  uint64_t carry = 0;  // order key of the record before this row
  for (int64_t i = g0;; i += 32) {
    const int64_t g = i + lane;
    Elt e{0, 0};
    uint64_t ok = 0;
    bool in = g < a.n;
    if (in) {
      e = ld_stream(a.src + g);
      ok = digit_key<ORD>(e.key, a.korder);
      in = (ok >> a.top_shift) == top0;
    }
    const unsigned out = ~__ballot_sync(0xffffffffu, in);
    const unsigned run = out ? (1u << (__ffs(out) - 1)) - 1 : 0xffffffffu;  // lanes before the bucket's end
    const bool mine = (run >> lane) & 1u;
    uint64_t prev = __shfl_up_sync(0xffffffffu, ok, 1);
    if (lane == 0) prev = carry;
    if (__any_sync(0xffffffffu, mine && ok < prev)) return false;
    if (mine) st_elt(a.dst + g, e);
    carry = __shfl_sync(0xffffffffu, ok, 31);
    if (run != 0xffffffffu) return true;
  }
}

template <bool ORD>
__global__ void __launch_bounds__(BK_THREADS, 2) bucket_sort_kernel(const BucketArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t s_bar;
  const Elt* s_raw = reinterpret_cast<const Elt*>(smem);
  unsigned* bits = reinterpret_cast<unsigned*>(smem + BK_SMEM_BITS);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int64_t t0 = (int64_t)blockIdx.x * BK_TILE;
  const int64_t w0 = t0 > 0 ? t0 - 1 : 0;
  const int64_t w1 = min(t0 + BK_TILE + BK_C, a.n);
  const int wlen = (int)(w1 - w0);
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_expect_tx(&s_bar, (unsigned)wlen * 16u);
    bulk_load(smem, a.src + w0, (unsigned)wlen * 16u, &s_bar);
  }
  __syncthreads();
  mbar_wait(&s_bar, 0);

  // boundary bits of window positions [own_lo, wlen]: a bucket starts at i (top differs from i - 1's, or global 0);
  // position wlen is a boundary when the window ends at n
  const int own_lo = (int)(t0 - w0);
  for (int wd = warp; wd < BK_WORDS; wd += BK_WARPS) {
    const int i = wd * 32 + lane;
    bool f = false;
    if (i >= own_lo && i < wlen) {
      const uint64_t top = digit_key<ORD>(s_raw[i].key, a.korder) >> a.top_shift;
      f = w0 + i == 0 || top != (digit_key<ORD>(s_raw[i - 1].key, a.korder) >> a.top_shift);
    } else if (i == wlen) {
      f = w1 == a.n;
    }
    const unsigned b = __ballot_sync(0xffffffffu, f);
    if (lane == 0) bits[wd] = b;
  }
  __syncthreads();

  const int own_end = (int)(min(t0 + BK_TILE, a.n) - w0);
  const int seg_lo = own_lo + warp * BK_SEG;
  const int seg_hi = min(seg_lo + BK_SEG, own_end);
  if (seg_lo >= seg_hi) return;
  int p = bk_find_first(bits, seg_lo, seg_hi - 1, lane);
  if (p < 0) return;  // no bucket starts here: the buckets around belong to other warps
  // end of the warp's last bucket; not within BK_C of seg_hi: that bucket is longer than BK_C
  // (a chunk ends at a boundary <= min(e_end, wlen))
  const int e_end = bk_find_first(bits, seg_hi, min(seg_hi + BK_C, wlen), lane);
  const int q_max = e_end < 0 ? wlen : e_end;

  uint64_t* keys = reinterpret_cast<uint64_t*>(smem + BK_SMEM_KEYS) + warp * BK_C;
  while (p < seg_hi) {
    const int q = bk_find_last(bits, p + 1, min(p + BK_C, q_max), lane);
    if (q < 0) {  // the bucket at p holds more than BK_C records, so it ends past seg_hi: the warp's last bucket
      if (!bk_long_bucket<ORD>(a, w0 + p, lane) && lane == 0) *a.overflow = 1u;
      return;
    }
    // the network sized to the chunk: a warp's last chunk is often a short remainder
    const int len = q - p;
    if (len <= 64) bk_sort_chunk<2, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
    else if (len <= 128) bk_sort_chunk<4, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
    else bk_sort_chunk<8, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
    p = q;
  }
}

}  // namespace lsb
