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
// chunk is sorted in the warp's registers (a bitonic network of 64, 128 or 256 keys: 2, 4 or 8 per lane), first by the
// 32-bit key (bk_sort_chunk32)
//   (ordinal << (24 - w) | prefix) << 8 | pos
// ordinal = index of the record's bucket in the chunk (monotone in top, so it stands for the top bits), w = the bits of
// the chunk's largest ordinal (0..8: a chunk of b buckets has ordinals 0..b - 1), prefix = the top 24 - w bits of the
// low 64 - 8k bits of order_key (all of them when they fit), pos = index in the chunk (equal keys keep their order).
// A chunk with padding has fewer than 32 * R records, so every pos, and with it the low byte of every real key, is at
// most 32 * R - 2 <= 254: the padding key 0xFFFFFFFF sorts after every record.  When the prefix drops low bits, two
// records of a bucket may share ordinal | prefix; the sorted ranks are then checked for such neighbours whose order
// keys differ, and a chunk that has one is sorted again by the 64-bit key (bk_sort_chunk)
//   ordinal << ord_shift | low << 8 | pos
// with the whole low part.  For k >= 2 and BK_C <= 256 that fills at most 64 bits, and a chunk with padding has fewer
// than 256 records, so its ordinals stay below 255 and the padding key ~0 sorts after every record.  Lane-major stores
// then write rank r of the chunk to chunk start + r.
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
  unsigned long long* prof;  // stage clocks, LSB_OP_PROF builds only (tools/bench_bucket.py)
};

// LSB_OP_PROF build (tools/ only): thread 0 of every CTA adds the clock64() delta since the previous stage mark to
// prof[BK_PROF0 + i] (so the chunk stages are those of warp 0's chunks), and lane 0 of every warp adds its chunk
// counts; the product build compiles none of it.
constexpr int BK_PROF0 = 40;
enum { BK_P_LOAD, BK_P_BITS, BK_P_KEYS, BK_P_NET, BK_P_TIES, BK_P_STORE, BK_P_FALLBACK, BK_P_LONG, BK_P_NSTAGE,
       BK_P_CTAS = BK_P_NSTAGE, BK_P_CHUNKS, BK_P_FALLBACKS, BK_P_LONGS, BK_NPROF };
#ifdef LSB_OP_PROF
#define BK_T(i)                                                                   \
  do {                                                                            \
    if (threadIdx.x == 0 && a.prof) {                                             \
      const long long now_ = clock64();                                           \
      atomicAdd(a.prof + BK_PROF0 + (i), (unsigned long long)(now_ - bk_prof_t)); \
      bk_prof_t = now_;                                                           \
    }                                                                             \
  } while (0)
#define BK_T_DECL long long bk_prof_t = clock64()
#define BK_T_ARG , long long& bk_prof_t
#define BK_T_PASS , bk_prof_t
#define BK_COUNT(i, v)                                                                         \
  do {                                                                                         \
    if (lane == 0 && a.prof && (v)) atomicAdd(a.prof + BK_PROF0 + (i), (unsigned long long)(v)); \
  } while (0)
#else
#define BK_T(i) do {} while (0)
#define BK_T_DECL
#define BK_T_ARG
#define BK_T_PASS
#define BK_COUNT(i, v) do {} while (0)
#endif

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

// ascending bitonic sort of 32 * R 32-bit keys, key (lane * R + r) in k[r], with every comparator ascending: each merge
// of two sorted runs of kk / 2 first compares key i with its mirror i ^ (kk - 1), then half-cleans with i ^ j, and the
// lower index always keeps the min.  Within a lane a compare-exchange is one unsigned min and one max; across lanes a
// key moves in one shuffle and the lane keeps the min or the max.
template <int R>
__device__ __forceinline__ void bk_bitonic32(uint32_t (&k)[R], int lane) {
#pragma unroll
  for (int kk = 2; kk <= 32 * R; kk <<= 1) {
#pragma unroll
    for (int j = kk >> 1; j > 0; j >>= 1) {
      const bool mirror = j == kk >> 1;  // partner i ^ (kk - 1), else i ^ j
      if (j >= R) {  // partner in lane ^ (kk / R - 1) or lane ^ (j / R)
        const int lj = mirror ? kk / R - 1 : j / R;
        const bool lower = (lane & (j / R)) == 0;
        uint32_t o[R];
#pragma unroll
        for (int r = 0; r < R; r++) o[r] = __shfl_xor_sync(0xffffffffu, k[mirror ? R - 1 - r : r], lj);
#pragma unroll
        for (int r = 0; r < R; r++) k[r] = lower ? min(k[r], o[r]) : max(k[r], o[r]);
      } else {  // partner in register r ^ (kk - 1) or r ^ j, same lane
#pragma unroll
        for (int r = 0; r < R; r++) {
          if (r & j) continue;
          const int q = mirror ? r ^ (kk - 1) : r | j;
          const uint32_t lo = min(k[r], k[q]), hi = max(k[r], k[q]);
          k[r] = lo;
          k[q] = hi;
        }
      }
    }
  }
}

// the chunk [p, p + len) of window positions, len <= 32 * R, sorted by its 32-bit chunk keys and stored to dst + w0 + p;
// false (nothing stored) when two records share ordinal | prefix but not their order keys: the prefix cannot order them
template <int R, bool ORD>
__device__ __forceinline__ bool bk_sort_chunk32(const BucketArgs& a, const Elt* s_raw, const unsigned* bits,
                                                unsigned char* perm, int p, int len, int64_t w0, int lane BK_T_ARG) {
  // record e = r * 32 + lane goes to k[r]: the network sorts whatever slots the keys start in
  int ord[R];
  int last = 0;  // the chunk's largest ordinal
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int e = r * 32 + lane;
    const bool start = e < len && e > 0 && bk_bit(bits, p + e);
    const unsigned b = __ballot_sync(0xffffffffu, start);
    ord[r] = last + __popc(b & (lanemask_lt() << 1 | 1u));
    last += __popc(b);
  }
  const int pw = 24 - (32 - __clz(last));        // prefix bits
  const int drop = max(a.top_shift - pw, 0);     // low bits the prefix leaves out
  uint32_t k[R];
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int e = r * 32 + lane;
    k[r] = ~0u;
    if (e < len) {
      const uint64_t low = digit_key<ORD>(s_raw[p + e].key, a.korder) & a.low_mask;
      k[r] = ((uint32_t)ord[r] << pw | (uint32_t)(low >> drop)) << 8 | (uint32_t)e;
    }
  }
  BK_T(BK_P_KEYS);
  bk_bitonic32<R>(k, lane);
  BK_T(BK_P_NET);
  if (drop) {
    // ranks lane * R + r and lane * R + r + 1, both records, with equal ordinal | prefix: equal order keys are in pos
    // order already, different ones need the whole low part
    const uint32_t next0 = __shfl_down_sync(0xffffffffu, k[0], 1);
    bool bad = false;
#pragma unroll
    for (int r = 0; r < R; r++) {
      const uint32_t nx = r + 1 < R ? k[r + 1] : next0;
      if (lane * R + r + 1 < len && (nx >> 8) == (k[r] >> 8))
        bad = bad || digit_key<ORD>(s_raw[p + (k[r] & 255)].key, a.korder) !=
                         digit_key<ORD>(s_raw[p + (nx & 255)].key, a.korder);
    }
    if (__any_sync(0xffffffffu, bad)) return false;
  }
  BK_T(BK_P_TIES);
  // chunk position of rank e: perm[e], R bytes per lane in one store
  if constexpr (R == 2) {
    reinterpret_cast<unsigned short*>(perm)[lane] = (unsigned short)__byte_perm(k[0], k[1], 0x0040);
  } else {
    uint32_t w[R / 4];
#pragma unroll
    for (int i = 0; i < R / 4; i++)
      w[i] = __byte_perm(__byte_perm(k[4 * i], k[4 * i + 1], 0x0040), __byte_perm(k[4 * i + 2], k[4 * i + 3], 0x0040), 0x5410);
    if constexpr (R == 4) reinterpret_cast<uint32_t*>(perm)[lane] = w[0];
    else reinterpret_cast<uint2*>(perm)[lane] = make_uint2(w[0], w[1]);
  }
  __syncwarp();
  Elt* out = a.dst + w0 + p;
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int e = r * 32 + lane;
    if (e < len) st_elt(out + e, s_raw[p + perm[e]]);
  }
  __syncwarp();
  BK_T(BK_P_STORE);
  return true;
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
  BK_T_DECL;

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
  BK_T(BK_P_LOAD);

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
  BK_T(BK_P_BITS);
  BK_COUNT(BK_P_CTAS, warp == 0);

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
  unsigned char* perm = reinterpret_cast<unsigned char*>(keys);
  int chunks = 0, fallbacks = 0;
  while (p < seg_hi) {
    const int q = bk_find_last(bits, p + 1, min(p + BK_C, q_max), lane);
    if (q < 0) {  // the bucket at p holds more than BK_C records, so it ends past seg_hi: the warp's last bucket
      if (!bk_long_bucket<ORD>(a, w0 + p, lane) && lane == 0) *a.overflow = 1u;
      BK_T(BK_P_LONG);
      BK_COUNT(BK_P_LONGS, 1);
      break;
    }
    // the network sized to the chunk: a warp's last chunk is often a short remainder; the 64-bit key when the prefix
    // of the 32-bit one leaves two records unordered
    const int len = q - p;
    bool done;
    if (len <= 64) done = bk_sort_chunk32<2, ORD>(a, s_raw, bits, perm, p, len, w0, lane BK_T_PASS);
    else if (len <= 128) done = bk_sort_chunk32<4, ORD>(a, s_raw, bits, perm, p, len, w0, lane BK_T_PASS);
    else done = bk_sort_chunk32<8, ORD>(a, s_raw, bits, perm, p, len, w0, lane BK_T_PASS);
    if (!done) {
      if (len <= 64) bk_sort_chunk<2, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
      else if (len <= 128) bk_sort_chunk<4, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
      else bk_sort_chunk<8, ORD>(a, s_raw, bits, keys, p, len, w0, lane);
      fallbacks++;
      BK_T(BK_P_FALLBACK);
    }
    chunks++;
    p = q;
  }
  BK_COUNT(BK_P_CHUNKS, chunks);
  BK_COUNT(BK_P_FALLBACKS, fallbacks);
}

}  // namespace lsb
