// lsb_kernels.cuh -- sm_100a device code of the LSD radix sort hot path.
//
// Reference path being replaced (citations relative to /root/reference/):
//   generator loop ............ mpi/mpi_lsbsort.cpp:650-656   -> generate_kernel
//   localShuffle count ........ mpi/mpi_lsbsort.cpp:226-229   -> digit_hist_kernel (lsb_onepass.cuh)
//   count transpose + scan .... mpi/mpi_lsbsort.cpp:327-479   -> scan kernels (digit-major, rank-minor)
//   localShuffle scatter ...... mpi/mpi_lsbsort.cpp:241-246   -> onepass_kernel (lsb_onepass.cuh), partition_kernel
//   pack / alltoallv / unpack . mpi/mpi_lsbsort.cpp:530-576   -> exchange_vr_kernel
//   verify .................... mpi/mpi_lsbsort.cpp:710-739   -> verify_kernel / checksum
//
// Everything here is integer/byte work bound by HBM (and NVLink for G > 1); no tensor cores.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lsb_keyorder.cuh"

namespace lsb {

typedef unsigned __int128 u128;

// What a digit is read from: the key itself (uint64 ascending, ORD = false: the kernels compile exactly as without key
// orders) or order_key(key, korder) (ORD = true: one instantiation serves every order, korder holds its flags).
template <bool ORD>
__device__ __forceinline__ uint64_t digit_key(uint64_t k, uint32_t korder) {
  return ORD ? order_key(k, korder) : k;
}

struct __align__(16) Elt {
  uint64_t key;
  uint64_t val;
};

// ------------------------------------------------------------------------------------
// memory helpers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ Elt ld_stream(const Elt* p) {
  Elt e;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(e.key), "=l"(e.val) : "l"(p));
  return e;
}
__device__ __forceinline__ uint64_t ld_stream_key(const Elt* p) {
  uint64_t k;
  asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(k) : "l"(p));
  return k;
}
__device__ __forceinline__ void st_elt(Elt* p, const Elt& e) {
  asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(e.key), "l"(e.val) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_gpu(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_gpu(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// ------------------------------------------------------------------------------------
// PCG64 (setseq_xsl_rr_128_64 with the default stream), the generator pcg64(myRank)
// of mpi/mpi_lsbsort.cpp:650-653.  Not vendored by the reference (mpi/getpcg.sh:3);
// restated from the published algorithm: 128-bit LCG, advance first, XSL-RR output.
// ------------------------------------------------------------------------------------
#define LSB_PCG_MULT_HI 2549297995355413924ULL
#define LSB_PCG_MULT_LO 4865540595714422341ULL
#define LSB_PCG_INC_HI 6364136223846793005ULL
#define LSB_PCG_INC_LO 1442695040888963407ULL

__host__ __device__ __forceinline__ u128 mk128(uint64_t hi, uint64_t lo) { return ((u128)hi << 64) | lo; }
__host__ __device__ __forceinline__ u128 pcg_mult() { return mk128(LSB_PCG_MULT_HI, LSB_PCG_MULT_LO); }
__host__ __device__ __forceinline__ u128 pcg_inc() { return mk128(LSB_PCG_INC_HI, LSB_PCG_INC_LO); }
__host__ __device__ __forceinline__ u128 pcg_seed(uint64_t seed) {
  return ((u128)seed + pcg_inc()) * pcg_mult() + pcg_inc();
}
__host__ __device__ __forceinline__ uint64_t pcg_output(u128 s) {
  uint64_t hi = (uint64_t)(s >> 64), lo = (uint64_t)s;
  unsigned rot = (unsigned)(hi >> 58);
  uint64_t x = hi ^ lo;
  return (x >> rot) | (x << ((64u - rot) & 63u));
}
// affine map x -> mult*x + plus that equals `delta` LCG steps (Brown's jump-ahead)
__host__ __device__ inline void pcg_jump_coeffs(u128 delta, u128& acc_mult, u128& acc_plus) {
  u128 cur_mult = pcg_mult(), cur_plus = pcg_inc();
  acc_mult = 1;
  acc_plus = 0;
  while (delta > 0) {
    if (delta & 1) {
      acc_mult *= cur_mult;
      acc_plus = acc_plus * cur_mult + cur_plus;
    }
    cur_plus = (cur_mult + 1) * cur_plus;
    cur_mult *= cur_mult;
    delta >>= 1;
  }
}

struct GenArgs {
  Elt* dst;             // shard base
  int64_t first_global; // global index of dst[0]
  int64_t count;        // elements of this shard (here)
  int64_t per_stream;   // ceil(n / R): slots per pcg stream
  uint64_t seed_base;
  uint64_t key_mask;
  int32_t and_draws;    // k
  // affine map for a jump of 32*k draws (one warp row)
  uint64_t row_mult_hi, row_mult_lo, row_plus_hi, row_plus_lo;
};

constexpr int GEN_ROWS = 64;       // rows of 32 elements per warp
constexpr int GEN_THREADS = 256;

// Warp w owns GEN_ROWS consecutive rows of 32 elements; lane l owns column l, so every
// store is a coalesced 512-byte row.  A lane walks its column with the precomputed
// 32*k-step affine map and only pays the O(log) jump-ahead when it (re)enters a stream.
__global__ void __launch_bounds__(GEN_THREADS) generate_kernel(const GenArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * GEN_THREADS + threadIdx.x) >> 5;
  const int64_t chunk0 = warp * (32 * GEN_ROWS);
  if (chunk0 >= a.count) return;
  const u128 mult = pcg_mult(), inc = pcg_inc();
  const u128 row_mult = mk128(a.row_mult_hi, a.row_mult_lo), row_plus = mk128(a.row_plus_hi, a.row_plus_lo);
  const int k = a.and_draws;
  u128 state = 0;
  int64_t stream_end = -1;  // global index where the current stream ends (exclusive)
  for (int t = 0; t < GEN_ROWS; t++) {
    const int64_t li = chunk0 + (int64_t)t * 32 + lane;
    if (li >= a.count) break;
    const int64_t gi = a.first_global + li;
    if (gi >= stream_end) {  // first row, or crossed into the next rank's stream
      const int64_t r = gi / a.per_stream;
      const int64_t j = gi - r * a.per_stream;
      u128 jm, jp;
      pcg_jump_coeffs((u128)j * (u128)k, jm, jp);
      state = jm * pcg_seed(a.seed_base + (uint64_t)r) + jp;
      stream_end = (r + 1) * a.per_stream;
    }
    u128 s = state;
    uint64_t key = ~0ULL;
    for (int d = 0; d < k; d++) {
      s = s * mult + inc;
      key &= pcg_output(s);
    }
    Elt e;
    e.key = key & a.key_mask;
    e.val = (uint64_t)gi;
    st_elt(a.dst + li, e);
    state = state * row_mult + row_plus;
  }
}

// ------------------------------------------------------------------------------------
// sub-digit counts for the two-step pass shape (localShuffle's count loop, mpi/mpi_lsbsort.cpp:
// 226-229, once for the whole sort): ONE read of the shard produces the 256-bin histograms of up to
// 16 sub-digits.  Block-private shared-memory histograms, coalesced 8-byte key loads with 4 loads in
// flight per thread, one global atomic per bin per CTA.  NSUB is a compile-time count so the per-key
// loop is fully unrolled; BYTES = the sub-digits are exactly bytes 0..NSUB-1 of the key (radix 8/16).
// Skew: when the whole warp agrees on the key's upper 32 bits (keys with few random bits), the
// sub-digits that live there are counted by one lane (+popc) instead of a 32-way same-address atomic.
// ------------------------------------------------------------------------------------
constexpr int HIST_THREADS = 512;
constexpr int HIST_MAX_SUB = 16;

struct HistArgs {
  const Elt* src;
  int64_t m;
  int32_t nsub;
  int32_t shift[HIST_MAX_SUB];
  uint32_t mask[HIST_MAX_SUB];
  unsigned long long* out;  // [nsub][256], accumulated with atomics (caller zeroes)
  uint32_t korder;          // key-order flags (ORD instantiations)
};

template <int NSUB, bool BYTES>
__device__ __forceinline__ void hist_key(unsigned* sh, uint64_t k, const int* shift, const unsigned* mask,
                                         unsigned active) {
  const int leader_lane = __ffs(active) - 1;
  const unsigned hi = (unsigned)(k >> 32);
  const bool hi_uniform = __all_sync(active, hi == __shfl_sync(active, hi, leader_lane));
  const bool leader = (int)(threadIdx.x & 31) == leader_lane;
#pragma unroll
  for (int s = 0; s < NSUB; s++) {
    const int sh_s = BYTES ? 8 * s : shift[s];
    const unsigned bin = BYTES ? (unsigned)(k >> (8 * s)) & 255u : (unsigned)(k >> sh_s) & mask[s];
    const bool in_hi = BYTES ? (s >= 4) : (sh_s >= 32);
    if (in_hi && hi_uniform) {
      if (leader) atomicAdd(sh + s * 256 + bin, (unsigned)__popc(active));
    } else {
      atomicAdd(sh + s * 256 + bin, 1u);
    }
  }
}

template <int NSUB, bool BYTES, bool ORD>
__global__ void __launch_bounds__(HIST_THREADS) subdigit_hist_kernel(const HistArgs a) {
  __shared__ unsigned sh[NSUB * 256];
  for (int i = threadIdx.x; i < NSUB * 256; i += HIST_THREADS) sh[i] = 0;
  int shift[NSUB];
  unsigned mask[NSUB];
#pragma unroll
  for (int s = 0; s < NSUB; s++) { shift[s] = a.shift[s]; mask[s] = a.mask[s]; }
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * HIST_THREADS;  // a multiple of 32
  int64_t i = (int64_t)blockIdx.x * HIST_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  constexpr int U = 4;
  // the unrolled loop runs only while the WHOLE warp is in range (full-mask shuffles inside)
  for (; (i - lane) + 31 + (U - 1) * stride < a.m; i += U * stride) {
    uint64_t k[U];
#pragma unroll
    for (int u = 0; u < U; u++) k[u] = digit_key<ORD>(ld_stream_key(a.src + i + u * stride), a.korder);
#pragma unroll
    for (int u = 0; u < U; u++) hist_key<NSUB, BYTES>(sh, k[u], shift, mask, 0xffffffffu);
  }
  for (; i < a.m; i += stride) {
    const unsigned active = __activemask();
    hist_key<NSUB, BYTES>(sh, digit_key<ORD>(ld_stream_key(a.src + i), a.korder), shift, mask, active);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < NSUB * 256; j += HIST_THREADS)
    if (sh[j]) atomicAdd(a.out + j, (unsigned long long)sh[j]);
}

// ------------------------------------------------------------------------------------
// scans
// ------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t warp_incl_scan(uint64_t v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint64_t o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += o;
  }
  return v;
}

// blockDim.x == 256: exclusive scan of one 256-bin histogram per block.
// out[b*257 + 0..255] = exclusive prefix, out[b*257 + 256] = total.
__global__ void __launch_bounds__(256) scan256_kernel(const unsigned long long* hist, int64_t* out) {
  __shared__ uint64_t wtot[8];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const uint64_t c = hist[(size_t)blockIdx.x * 256 + t];
  const uint64_t incl = warp_incl_scan(c);
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  uint64_t off = 0;
  for (int i = 0; i < w; i++) off += wtot[i];
  out[(size_t)blockIdx.x * 257 + t] = (int64_t)(off + incl - c);
  if (t == 255) out[(size_t)blockIdx.x * 257 + 256] = (int64_t)(off + incl);
}

// The reference's copyCountsToGlobalCounts + exclusiveScan + copyStartsFromGlobalStarts
// (mpi/mpi_lsbsort.cpp:327-479) in one kernel: exclusive scan of counts[g][d] in
// digit-major, rank-minor order (dstGlobalIdx = d*R + rank, :350) and extraction of this
// rank's column: mybase[d] = GlobalStarts[d*G + my].  Also the elements this rank sends to
// each destination shard (sendCounts, :553-554).  One CTA of 1024 threads; the table is
// at most 65536 x 8 counts.
struct GlobalScanArgs {
  const unsigned long long* counts;  // [G][nb]
  int32_t nb;
  int32_t G;
  int32_t my;
  int64_t per;                       // destination shard size
  int64_t* mybase;                   // [nb]
  unsigned long long* sent;          // [G] (caller zeroes) or nullptr
};

__global__ void __launch_bounds__(1024) global_scan_kernel(const GlobalScanArgs a) {
  __shared__ uint64_t wtot[32];
  __shared__ unsigned long long s_sent[8];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  if (t < 8) s_sent[t] = 0;
  const int chunk = (a.nb + 1023) / 1024;
  const int d0 = t * chunk, d1 = min(d0 + chunk, a.nb);
  uint64_t local = 0;
  for (int d = d0; d < d1; d++)
    for (int g = 0; g < a.G; g++) local += a.counts[(size_t)g * a.nb + d];
  const uint64_t incl = warp_incl_scan(local);
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  uint64_t run = incl - local;
  for (int i = 0; i < w; i++) run += wtot[i];
  unsigned long long sent[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int d = d0; d < d1; d++)
    for (int g = 0; g < a.G; g++) {
      const uint64_t c = a.counts[(size_t)g * a.nb + d];
      if (g == a.my) {
        a.mybase[d] = (int64_t)run;
        if (c && a.sent) {  // split [run, run+c) over destination shards
          uint64_t b = run, e = run + c;
          while (b < e) {
            const uint64_t r = b / (uint64_t)a.per;
            const uint64_t lim = (r + 1) * (uint64_t)a.per;
            const uint64_t x = e < lim ? e : lim;
            sent[r] += x - b;
            b = x;
          }
        }
      }
      run += c;
    }
  if (a.sent) {
    for (int g = 0; g < a.G; g++)
      if (sent[g]) atomicAdd(&s_sent[g], sent[g]);
    __syncthreads();
    if (t < a.G) a.sent[t] = s_sent[t];
  }
}

// ------------------------------------------------------------------------------------
// tile machinery shared by partition_kernel (below) and onepass_kernel (lsb_onepass.cuh):
// a tile of elements sits in shared memory (pulled in by the TMA engine: cp.async.bulk with
// mbarrier completion, so no registers hold elements), is ranked stably by an 8-bit key
// with warp ballots, and is written out through a 2-byte permutation perm[slot] = index.
// ------------------------------------------------------------------------------------
template <int THREADS_, int IPT_, int MINB_>
struct PartCfg {
  static constexpr int THREADS = THREADS_;
  static constexpr int WARPS = THREADS_ / 32;
  static constexpr int LOG_WARPS = THREADS_ == 1024 ? 5 : THREADS_ == 512 ? 4 : THREADS_ == 256 ? 3 : THREADS_ == 128 ? 2 : -1;
  static constexpr int IPT = IPT_;
  static constexpr int MINB = MINB_;
  static constexpr int TILE = THREADS_ * IPT_;
  // raw tile | perm (u16) | per-warp histograms (u16) | bin -> destination offset (i64)
  static constexpr int SMEM_RAW = 0;
  static constexpr int SMEM_PERM = SMEM_RAW + TILE * 16;
  static constexpr int SMEM_WHIST = SMEM_PERM + TILE * 2;
  static constexpr int SMEM_BINDST = SMEM_WHIST + WARPS * 256 * 2;
  static constexpr int SMEM = SMEM_BINDST + 256 * 8;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_init_nofence(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  while (!mbar_try(bar, parity)) {}
}
// global -> shared bulk copy on the TMA engine; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// L2 eviction-priority policies and a bulk load that carries one
__device__ __forceinline__ uint64_t l2_policy(int kind) {  // 0 normal, 1 evict_first, 2 evict_last
  uint64_t p;
  if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_load_hint(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar,
                                               uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
// global -> L2 only (no destination, no completion): bytes % 16 == 0, address 16-byte aligned
__device__ __forceinline__ void bulk_prefetch_l2(const void* src_gmem, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}

// lanes of `vmask` whose 8-bit `bin` equals mine: 8 ballots (hardware match.any, whole or per
// nibble, measured 30-40 % slower: its cost grows with the number of distinct values in the
// warp, and a row of 32 bins is mostly distinct)
template <bool FULL>
__device__ __forceinline__ unsigned match_bin(unsigned vmask, unsigned bin) {
  unsigned peers = vmask;
  if (FULL) {
#pragma unroll
    for (int b = 0; b < 8; b++) {
      // 4 SASS instructions per bit (the C++ form below compiles to 6-7): bit test -> predicate,
      // ballot, select 0 / ~0 on the same predicate, peers &= ballot ^ select
      unsigned bal;
      asm("{\n\t.reg .pred p;\n\t.reg .b32 t, m;\n\t"
          "and.b32 t, %2, %3;\n\t"
          "setp.ne.u32 p, t, 0;\n\t"
          "vote.sync.ballot.b32 %1, p, 0xffffffff;\n\t"
          "selp.b32 m, 0, -1, p;\n\t"
          "lop3.b32 %0, %0, %1, m, 0x60;\n\t}"
          : "+r"(peers), "=r"(bal)
          : "r"(bin), "r"(1u << b));
      (void)bal;
    }
  } else {
#pragma unroll
    for (int b = 0; b < 8; b++) {
      const bool bit = (bin & (1u << b)) != 0;
      const unsigned bal = __ballot_sync(vmask, bit);
      peers &= bal ^ (bit ? 0u : 0xffffffffu);
    }
  }
  return peers;
}

// How a tile of `count` elements is dealt to the warps: rows of 32 elements in contiguous blocks
// (warp order == index order, which the stable per-warp offsets need), as evenly as the count
// allows, so a partly filled tile keeps every warp busy.  Only the last row of a tile can be
// partial; it belongs to the last warp that has rows and is handled outside the unrolled loop.
struct RowPlan {
  int row0;      // first row of this warp
  int nfull;     // full rows of this warp
  int ptail;     // elements in this warp's partial row (0 = none); the row index is row0 + nfull
};
template <class C>
__device__ __forceinline__ RowPlan row_plan(int count) {
  const int warp = threadIdx.x >> 5;
  const int full = count >> 5, tail = count & 31;
  const int rows = full + (tail ? 1 : 0);
  const int base = rows / C::WARPS, extra = rows % C::WARPS;  // WARPS is a power of two
  RowPlan r;
  r.row0 = warp * base + min(warp, extra);
  const int mine = base + (warp < extra ? 1 : 0);
  r.nfull = max(0, min(mine, full - r.row0));
  r.ptail = (mine > r.nfull) ? tail : 0;
  return r;
}

// 8-bit digit of an element in shared memory; BYTE: the digit is exactly byte `shift / 8` of the key (raw key bits,
// so never under a key order)
template <bool BYTE, bool ORD>
__device__ __forceinline__ unsigned tile_bin(const Elt* e, int shift, unsigned mask, uint32_t korder) {
  static_assert(!(BYTE && ORD), "the byte path reads the raw key");
  if (BYTE) return reinterpret_cast<const unsigned char*>(e)[shift >> 3];
  return (unsigned)(digit_key<ORD>(e->key, korder) >> shift) & mask;
}

// Stable ranks, step 1: every element's rank among the elements of its bin that precede it IN ITS
// WARP's rows (8 ballots per row find the peers; a per-warp counter per bin runs over the rows).
// On return info[j] = bin | rank << 8 for row j, and the warp's counters hold its counts per bin --
// no separate counting pass over the tile.  s_whist must be zero on entry.
template <class C, bool FULL, bool BYTE, bool ORD>
__device__ __forceinline__ void op_rank(const Elt* __restrict__ s_raw, const RowPlan& rp, int shift, unsigned mask,
                                        uint32_t korder, unsigned short* __restrict__ s_whist, unsigned (&info)[C::IPT],
                                        unsigned& info_p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned short* wh = s_whist + warp * 256;
  const unsigned lt = lanemask_lt();
  const Elt* row = s_raw + (FULL ? warp * (32 * C::IPT) : rp.row0 * 32) + lane;
  // all digits first: the loads must not sit inside the serial chain of counter updates below
#pragma unroll
  for (int j = 0; j < C::IPT; j++)
    info[j] = (FULL || j < rp.nfull) ? tile_bin<BYTE, ORD>(row + j * 32, shift, mask, korder) : 0;
  info_p = (!FULL && lane < rp.ptail) ? tile_bin<BYTE, ORD>(row + rp.nfull * 32, shift, mask, korder) : 0;
#pragma unroll
  for (int j = 0; j < C::IPT; j++) {
    if (FULL || j < rp.nfull) {
      const unsigned bin = info[j];
      const unsigned peers = match_bin<true>(0xffffffffu, bin);
      const unsigned old = wh[bin];
      __syncwarp();
      if ((peers & lt) == 0) wh[bin] = (unsigned short)(old + __popc(peers));
      __syncwarp();
      info[j] = bin | ((old + __popc(peers & lt)) << 8);
    }
  }
  if (!FULL && rp.ptail) {  // warp-uniform
    const bool valid = lane < rp.ptail;
    const unsigned vmask = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      const unsigned bin = info_p;
      const unsigned peers = match_bin<false>(vmask, bin);
      const unsigned old = wh[bin];
      __syncwarp(vmask);
      if ((peers & lt) == 0) wh[bin] = (unsigned short)(old + __popc(peers));
      __syncwarp(vmask);
      info_p = bin | ((old + __popc(peers & lt)) << 8);
    }
  }
}

// Step 2, threads 0..255 only (bin = tid): tile total of the bin, its start inside the sorted tile,
// and each warp's base slot for the bin written back over the warp's count.  Uses named barrier 1.
template <class C>
__device__ __forceinline__ void op_scan(unsigned short* s_whist, unsigned* s_wtot, unsigned& tile_count,
                                        unsigned& binstart) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned wc[C::WARPS];
  tile_count = 0;
#pragma unroll
  for (int w = 0; w < C::WARPS; w++) {
    wc[w] = s_whist[w * 256 + tid];
    tile_count += wc[w];
  }
  unsigned incl = tile_count;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) s_wtot[warp] = incl;
  asm volatile("bar.sync 1, 256;" ::: "memory");
  binstart = incl - tile_count;
  for (int i = 0; i < warp; i++) binstart += s_wtot[i];
  unsigned run = binstart;
#pragma unroll
  for (int w = 0; w < C::WARPS; w++) {
    s_whist[w * 256 + tid] = (unsigned short)run;
    run += wc[w];
  }
}

// Step 3: slot = warp base of the bin + rank; the sorted order as a permutation perm[slot] = index
template <class C, bool FULL>
__device__ __forceinline__ void op_perm(const RowPlan& rp, const unsigned short* s_whist, unsigned short* s_perm,
                                        const unsigned (&info)[C::IPT], unsigned info_p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned short* wh = s_whist + warp * 256;
  const int idx0 = (FULL ? warp * (32 * C::IPT) : rp.row0 * 32) + lane;
#pragma unroll
  for (int j = 0; j < C::IPT; j++)
    if (FULL || j < rp.nfull) s_perm[wh[info[j] & 255u] + (info[j] >> 8)] = (unsigned short)(idx0 + j * 32);
  if (!FULL && lane < rp.ptail) s_perm[wh[info_p & 255u] + (info_p >> 8)] = (unsigned short)(idx0 + rp.nfull * 32);
}

// ------------------------------------------------------------------------------------
// partition kernel: one stable counting-sort step on a digit of <= 8 bits, HBM -> HBM
// (localShuffle's scatter, mpi/mpi_lsbsort.cpp:241-246, for the narrow digits of a radix
// sweep; wider digits go through onepass_kernel).  One CTA = one tile, taken in input order
// by a dynamic tile id so that predecessors are always resident:
//   1. bulk-load the tile; 2. early per-warp counts -> tile totals published for the decoupled
//   look-back before the ranking starts; 3. stable ranks; 4. look-back over 64-bit {tag, count}
//   words, 4 predecessor tiles per round trip (the tag is a per-launch generation, so the words
//   are never cleared); 5. consecutive threads write consecutive slots of a bin's run.
// ------------------------------------------------------------------------------------
constexpr int PT_LB_WINDOW = 4;
constexpr int PT_MAX_CHUNKS = 16;
constexpr uint64_t LB_VALUE_MASK = (1ULL << 56) - 1;

struct PartArgs {
  const Elt* src;
  int32_t shift;
  uint32_t mask;
  int32_t seg_bits;                // nseg = 1 << seg_bits
  const int64_t* seg_start;        // [nseg + 1] element offsets into src
  const uint32_t* seg_tile_start;  // [nseg + 1] tile-index prefix
  const int64_t* bases;            // [(bin << seg_bits) | seg]: global output index of this shard's
                                   // first element of (seg, bin)
  uint64_t* lookback;              // [tiles][256]
  uint32_t* tile_counter;
  uint64_t tag_agg;                // (2*gen+1) << 56
  uint64_t tag_inc;                // (2*gen+2) << 56
  int64_t per;                     // destination shard size (global index / per = shard)
  int32_t world;
  Elt* dst[8];                     // destination shard base pointers (peer-mapped for g != my)
  unsigned long long* prof;        // stage clocks, LSB_OP_PROF builds only (tools/prof_stages.py)
  // direct mode (one segment known to the host): tile = blockIdx.x over src[d_begin, d_end); no ticket,
  // no segment table reads -- the bulk load is issued by the CTA's first instructions
  int32_t direct;
  int32_t log_chunks;              // log2 of the number of bulk copies a tile arrives in (pieces of whole warps' rows)
  int64_t d_begin, d_end;
  int32_t pf_tiles;                // L2PF: tile blockIdx.x + pf_tiles is pulled into L2 when this tile starts
  uint32_t korder;                 // key-order flags (ORD instantiations)
};

// L2PF (compile-time; lsb_tune "pt_variant" 1 = default, 0 = off): in direct mode the CTA of tile t also starts a bulk
// L2 prefetch of tile t + pf_tiles, so the tile load of the CTA that gets that tile a few microseconds later is an L2 hit:
// the HBM queueing moves off the CTA's serial path (7.09 -> 6.48 ms per launch at 2^30) and DRAM traffic is unchanged as
// long as the lines survive in L2 until then (distance 74..148 tiles; at 296 half the gain is gone, at 592 it is a loss).
// Two more variants were A/B-measured at commit a1530c7 and removed: the first look-back window loaded before the ranking
// phase (+3 % time) and evict_first tile loads (no gain), profiles/r2_final_sweep.log.

// LSB_OP_PROF build (tools/ only): thread 0 of every CTA adds the clock64() delta since the previous
// stage mark to prof[PT_PROF0 + i]; the product build compiles none of it.
constexpr int PT_PROF0 = 24, PT_PROF_TILES = 39;
#ifdef LSB_OP_PROF
#define PT_T(i)                                                                        \
  do {                                                                                 \
    if (threadIdx.x == 0 && a.prof) {                                                  \
      const long long now_ = clock64();                                                \
      atomicAdd(a.prof + PT_PROF0 + (i), (unsigned long long)(now_ - pt_prof_t));      \
      pt_prof_t = now_;                                                                \
    }                                                                                  \
  } while (0)
#define PT_T_DECL long long pt_prof_t
#define PT_T_ARG , long long pt_prof_t
#define PT_T_PASS , pt_prof_t
#else
#define PT_T(i) do {} while (0)
#define PT_T_DECL
#define PT_T_ARG
#define PT_T_PASS
#endif

// (round 1's kernel, kept as measured: a leaner restatement on the helpers above ran 7 % slower)
template <class C, bool FULL, bool ORD>
__device__ __forceinline__ void partition_tile(const PartArgs& a, unsigned char* smem, uint64_t* s_bar,
                                               unsigned* s_wtot, int tile, int seg, int count, bool first,
                                               int first_tile PT_T_ARG) {
  Elt* s_raw = reinterpret_cast<Elt*>(smem + C::SMEM_RAW);
  unsigned short* s_perm = reinterpret_cast<unsigned short*>(smem + C::SMEM_PERM);
  unsigned short* s_whist = reinterpret_cast<unsigned short*>(smem + C::SMEM_WHIST);
  long long* s_bindst = reinterpret_cast<long long*>(smem + C::SMEM_BINDST);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  {  // chunked load: wait only for the piece of the tile that holds this warp's rows
    const int lg = a.log_chunks;
    const int chunk = warp >> (C::LOG_WARPS - lg);
    if (chunk == 0 || chunk * (C::TILE >> lg) < count) mbar_wait(s_bar + chunk, 0);
  }
  PT_T(2);

  // ---- bins of my elements (warp-striped rows), early per-warp counts ----
  const int idx0 = warp * (32 * C::IPT) + lane;
  unsigned bins[C::IPT];
  unsigned* wh32 = reinterpret_cast<unsigned*>(s_whist + warp * 256);
#pragma unroll
  for (int j = 0; j < C::IPT; j++) {
    const int idx = idx0 + j * 32;
    bins[j] = 0;
    if (FULL || idx < count) {
      const unsigned bin = (unsigned)(digit_key<ORD>(s_raw[idx].key, a.korder) >> a.shift) & a.mask;
      bins[j] = bin;
      atomicAdd(wh32 + (bin >> 1), 1u << ((bin & 1u) * 16));
    }
  }
  __syncthreads();
  PT_T(3);

  // ---- per bin: tile total (published at once), exclusive over warps, start inside the tile ----
  unsigned tile_count = 0, binstart = 0;
  uint64_t* my_state = nullptr;
  long long my_base = 0;
  if (tid < 256) {
    my_state = a.lookback + (size_t)tile * 256 + tid;
    my_base = a.bases[((size_t)tid << a.seg_bits) | (unsigned)seg];  // early: its latency hides under the scan
    unsigned wc[C::WARPS];
#pragma unroll
    for (int w = 0; w < C::WARPS; w++) {
      wc[w] = s_whist[w * 256 + tid];
      tile_count += wc[w];
    }
    st_relaxed_gpu(my_state, (first ? a.tag_inc : a.tag_agg) | (uint64_t)tile_count);
    unsigned incl = tile_count;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) s_wtot[warp] = incl;
    asm volatile("bar.sync 1, 256;" ::: "memory");  // only the 8 scanning warps
    binstart = incl - tile_count;
    for (int i = 0; i < warp; i++) binstart += s_wtot[i];
    unsigned run = binstart;
#pragma unroll
    for (int w = 0; w < C::WARPS; w++) {
      s_whist[w * 256 + tid] = (unsigned short)run;
      run += wc[w];
    }
  }
  __syncthreads();
  PT_T(4);

  // ---- stable ranks: slot of each element inside the tile, written as a permutation ----
  {
    unsigned short* wh = s_whist + warp * 256;
    const unsigned lt = lanemask_lt();
#pragma unroll
    for (int j = 0; j < C::IPT; j++) {
      const int idx = idx0 + j * 32;
      const bool valid = FULL || idx < count;
      const unsigned vmask = FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid);
      if (valid) {
        const unsigned bin = bins[j];
        const unsigned peers = match_bin<FULL>(vmask, bin);
        const unsigned old = wh[bin];
        __syncwarp(vmask);
        if ((peers & lt) == 0) wh[bin] = (unsigned short)(old + __popc(peers));
        __syncwarp(vmask);
        s_perm[old + __popc(peers & lt)] = (unsigned short)idx;
      }
    }
  }

  PT_T(5);
  // ---- decoupled look-back: exclusive prefix of this bin over earlier tiles of the segment ----
  // A window of PT_LB_WINDOW predecessor words is fetched per round trip: with hundreds of tiles
  // in flight the walk is ~10 tiles deep, and one dependent L2 access per tile would dominate.
  if (tid < 256) {
    uint64_t excl = 0;
    if (!first) {
      int look = tile - 1;
      bool done = false;
      while (!done) {
#ifdef LSB_OP_PROF
        if (tid == 0 && a.prof) atomicAdd(a.prof + PT_PROF0 + 10, 1ULL);
#endif
        uint64_t v[PT_LB_WINDOW];
#pragma unroll
        for (int i = 0; i < PT_LB_WINDOW; i++) {
          const int t = look - i;
          v[i] = (t >= first_tile) ? ld_relaxed_gpu(a.lookback + (size_t)t * 256 + tid) : 0;
        }
        int used = 0;
#pragma unroll
        for (int i = 0; i < PT_LB_WINDOW; i++) {
          if (!done && used == i) {
            const uint64_t tag = v[i] & ~LB_VALUE_MASK;
            if (tag == a.tag_inc) { excl += v[i] & LB_VALUE_MASK; done = true; }
            else if (tag == a.tag_agg) { excl += v[i] & LB_VALUE_MASK; used = i + 1; }
          }
        }
        look -= used;
        if (!done && used == 0) __nanosleep(20);
      }
      st_relaxed_gpu(my_state, a.tag_inc | (excl + tile_count));
    }
    s_bindst[tid] = my_base + (long long)excl - (long long)binstart;
  }
  PT_T(6);
  __syncthreads();
  PT_T(7);

  // ---- write: consecutive threads -> consecutive slots of a bin's run ----
#pragma unroll
  for (int k = 0; k < C::IPT; k++) {
    const int p = k * C::THREADS + tid;
    const bool valid = FULL || p < count;
    Elt el;
    el.key = 0;
    el.val = 0;
    if (valid) {
      el = s_raw[s_perm[p]];
      const unsigned bin = (unsigned)(digit_key<ORD>(el.key, a.korder) >> a.shift) & a.mask;
      const long long g = s_bindst[bin] + p;
      Elt* out;
      if (a.world == 1) {
        out = a.dst[0] + g;
      } else {
        int r = 0;
        for (int q = 1; q < a.world; q++) r += (g >= (long long)q * a.per);
        out = a.dst[r] + (g - (long long)r * a.per);
      }
      st_elt(out, el);
    }
  }
  PT_T(8);
#ifdef LSB_OP_PROF
  if (threadIdx.x == 0 && a.prof) atomicAdd(a.prof + PT_PROF_TILES, 1ULL);
#endif
}

// one thread: arm the mbarriers and start the bulk copies of a tile of `cnt` elements; the tile arrives as
// 1 << log_chunks equal pieces so that a warp starts on its rows as soon as ITS piece has landed
template <class C>
__device__ __forceinline__ void partition_issue_load(const PartArgs& a, unsigned char* smem, uint64_t* s_bar, long long begin, int cnt) {
  static_assert((1 << C::LOG_WARPS) == C::WARPS && C::WARPS <= PT_MAX_CHUNKS, "a piece is a whole number of warps' rows");
  const int lg = a.log_chunks, nch = 1 << lg, ch = C::TILE >> lg;
  for (int q = 0; q < nch; q++) mbar_init_nofence(s_bar + q, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  for (int q = 0; q < nch; q++) {
    const int n = min(ch, cnt - q * ch);
    if (n > 0) {
      mbar_expect_tx(s_bar + q, (unsigned)n * 16u);
      bulk_load(smem + C::SMEM_RAW + (size_t)q * ch * 16, a.src + begin + q * ch, (unsigned)n * 16u, s_bar + q);
    }
  }
}

template <class C, bool L2PF, bool ORD>
__global__ void __launch_bounds__(C::THREADS, C::MINB) partition_kernel(const PartArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t s_bar[PT_MAX_CHUNKS];
  __shared__ int s_tile, s_seg, s_count, s_first, s_first_tile;
  __shared__ unsigned s_wtot[8];

  const int tid = threadIdx.x;
  const int nseg = 1 << a.seg_bits;
#ifdef LSB_OP_PROF
  PT_T_DECL = clock64();
#endif

  if (a.direct) {
    // tile ids in launch order (the hardware dispatches CTAs of a 1-D grid in blockIdx order, so every
    // predecessor a look-back waits for is resident or done): the load is in flight before anything else
    const long long begin = a.d_begin + (long long)blockIdx.x * C::TILE;
    const long long left = a.d_end - begin;
    const int cnt = (int)(left < C::TILE ? left : C::TILE);
    if (tid == 0) partition_issue_load<C>(a, smem, s_bar, begin, cnt);
    if constexpr (L2PF) {
      if (tid == 0) {
        const long long pb = begin + (long long)a.pf_tiles * C::TILE;
        const long long pl = a.d_end - pb;
        if (pl > 0) bulk_prefetch_l2(a.src + pb, (unsigned)(pl < C::TILE ? pl : C::TILE) * 16u);
      }
    }
    for (int i = tid; i < C::WARPS * 128; i += C::THREADS)
      reinterpret_cast<unsigned*>(smem + C::SMEM_WHIST)[i] = 0;
    __syncthreads();
    PT_T(0);
    PT_T(1);
    if (cnt == C::TILE)
      partition_tile<C, true, ORD>(a, smem, s_bar, s_wtot, (int)blockIdx.x, 0, cnt, blockIdx.x == 0, 0 PT_T_PASS);
    else
      partition_tile<C, false, ORD>(a, smem, s_bar, s_wtot, (int)blockIdx.x, 0, cnt, blockIdx.x == 0, 0 PT_T_PASS);
    return;
  }
  if (tid == 0) {
    const unsigned t = atomicAdd(a.tile_counter, 1u);
    s_tile = (t < a.seg_tile_start[nseg]) ? (int)t : -1;
    s_seg = 0;
  }
  // zero the packed per-warp histograms (WARPS*256 u16)
  for (int i = tid; i < C::WARPS * 128; i += C::THREADS)
    reinterpret_cast<unsigned*>(smem + C::SMEM_WHIST)[i] = 0;
  __syncthreads();
  PT_T(0);
  const int tile = s_tile;
  if (tile < 0) return;
  // which segment owns this tile: the one with first_tile <= tile < next first_tile
  if (nseg > 1) {
    if (tid < nseg) {
      const unsigned f = a.seg_tile_start[tid], l = a.seg_tile_start[tid + 1];
      if (f <= (unsigned)tile && (unsigned)tile < l) s_seg = tid;
    }
    __syncthreads();
  }
  if (tid == 0) {
    const int sg = s_seg;
    const unsigned t_in = (unsigned)tile - a.seg_tile_start[sg];
    const long long begin = a.seg_start[sg] + (long long)t_in * C::TILE;
    const long long left = a.seg_start[sg + 1] - begin;
    const int cnt = (int)(left < C::TILE ? left : C::TILE);
    s_count = cnt;
    s_first = (t_in == 0);
    s_first_tile = (int)a.seg_tile_start[sg];
    partition_issue_load<C>(a, smem, s_bar, begin, cnt);
  }
  __syncthreads();
  PT_T(1);
  const int count = s_count;
  if (count == C::TILE)
    partition_tile<C, true, ORD>(a, smem, s_bar, s_wtot, tile, s_seg, count, s_first, s_first_tile PT_T_PASS);
  else
    partition_tile<C, false, ORD>(a, smem, s_bar, s_wtot, tile, s_seg, count, s_first, s_first_tile PT_T_PASS);
}

// ------------------------------------------------------------------------------------
// exchange kernel (G > 1): the pack / MPI_Alltoallv / unpack of mpi/mpi_lsbsort.cpp:530-576
// as ONE pass over the shard once it is sorted by the full digit.  Element i of digit d goes to
// global index mybase[d] + (i - localbase[d]) (== `starts[bucket]++`, :550-552) and is stored
// straight into the owning GPU's shard (16 bytes on the wire, not the reference's 24).  A run
// (digit, this GPU) is contiguous on both sides, so the NVLink stores are long aligned bursts:
// measured 716 GB/s per direction for runs >= 128 B, against 220-620 GB/s (shard-size dependent:
// TLB set conflicts on cross-process peer mappings) when the 22-element runs of the scatter
// kernel are stored remotely (tools/p2p_bench.cu, tools/p2p_ipc_bench.cu).
// ------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------
// Pipelined multi-GPU pass ("virtual ranks"): every shard is cut into V contiguous parts and
// part q of GPU g acts as rank g*V+q of the reference's algorithm (its order is the global
// index order, so the result is unchanged).  Once the counts of the pass's full digit are known
// for every virtual rank BEFORE the pass starts, part q can be sorted locally and exchanged
// while part q+1 is being sorted: the NVLink time hides the local HBM time.  The counts of
// pass p+1 are produced by the exchange kernel of pass p (one L2 atomic per element, hidden
// under the NVLink time), per destination GPU and destination part.
// ------------------------------------------------------------------------------------

// global_scan_kernel for virtual ranks: counts[vr][d] (u32), scan in digit-major, virtual-rank-minor
// order; mybase[q][d] for this GPU's V parts (vr = first_vr + q), sent[] summed over the parts.
// Three small launches so that every pass over the [GV][nb] table is coalesced and spread over many
// CTAs: per-digit totals, exclusive scan of the totals (global_scan_kernel with G = 1), placement.
struct VrScanArgs {
  const unsigned* counts;  // [GV][nb]
  int32_t nb, GV, first_vr, V, G;
  int64_t per;             // destination shard size
  unsigned long long* totals;  // [nb] scratch: sum over virtual ranks
  const int64_t* digit_base;   // [nb] exclusive scan of totals
  int64_t* mybase;         // [V][nb]
  unsigned long long* sent;  // [G], caller zeroes (may be null)
};

__global__ void __launch_bounds__(256) vr_totals_kernel(const VrScanArgs a) {
  const int d = blockIdx.x * 256 + threadIdx.x;
  if (d >= a.nb) return;
  unsigned long long t = 0;
  for (int vr = 0; vr < a.GV; vr++) t += a.counts[(size_t)vr * a.nb + d];
  a.totals[d] = t;
}

__global__ void __launch_bounds__(256) vr_place_kernel(const VrScanArgs a) {
  __shared__ unsigned long long s_sent[8];
  if (threadIdx.x < 8) s_sent[threadIdx.x] = 0;
  __syncthreads();
  const int d = blockIdx.x * 256 + threadIdx.x;
  if (d < a.nb) {
    uint64_t run = (uint64_t)a.digit_base[d];
    for (int vr = 0; vr < a.GV; vr++) {
      const uint64_t c = a.counts[(size_t)vr * a.nb + d];
      const int q = vr - a.first_vr;
      if (q >= 0 && q < a.V) {
        a.mybase[(size_t)q * a.nb + d] = (int64_t)run;
        if (c && a.sent) {
          uint64_t b = run, e = run + c;
          while (b < e) {
            const uint64_t r = b / (uint64_t)a.per;
            const uint64_t lim = (r + 1) * (uint64_t)a.per;
            const uint64_t x = e < lim ? e : lim;
            atomicAdd(&s_sent[r], (unsigned long long)(x - b));
            b = x;
          }
        }
      }
      run += c;
    }
  }
  __syncthreads();
  if (a.sent && threadIdx.x < a.G && s_sent[threadIdx.x]) atomicAdd(a.sent + threadIdx.x, s_sent[threadIdx.x]);
}

// one block per part: where each digit's run starts inside the sorted part (localbase), and the
// bases of the two local counting-sort steps (sub-digit histograms folded out of the dense counts)
struct PartPrepArgs {
  const unsigned* counts;  // [V][nb] this GPU's parts, or
  const unsigned long long* counts64;  // [nb] (one part: the whole shard) when counts == nullptr
  int32_t nb, lo_bits, hi_bits;
  int64_t* localbase;      // [V][nb]
  int64_t* bases;          // [V][2][257]: exclusive scans of the low / high sub-digit counts (+ total)
};

__global__ void __launch_bounds__(1024) part_prep_kernel(const PartPrepArgs a) {
  __shared__ uint64_t wtot[32];
  __shared__ unsigned long long s_lo[256], s_hi[256];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const unsigned* c32 = a.counts ? a.counts + (size_t)blockIdx.x * a.nb : nullptr;
  auto cnt = [&](int d) -> unsigned long long { return c32 ? (unsigned long long)c32[d] : a.counts64[d]; };
  int64_t* lb = a.localbase + (size_t)blockIdx.x * a.nb;
  if (t < 256) { s_lo[t] = 0; s_hi[t] = 0; }
  __syncthreads();
  const int chunk = (a.nb + 1023) / 1024;
  const int d0 = t * chunk, d1 = min(d0 + chunk, a.nb);
  const unsigned lo_mask = (1u << a.lo_bits) - 1;
  uint64_t local = 0;
  for (int d = d0; d < d1; d++) {
    const unsigned long long v = cnt(d);
    local += v;
    if (v) {
      if (a.lo_bits) atomicAdd(&s_lo[d & lo_mask], v);
      atomicAdd(&s_hi[d >> a.lo_bits], v);
    }
  }
  const uint64_t incl = warp_incl_scan(local);
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  uint64_t run = incl - local;
  for (int i = 0; i < w; i++) run += wtot[i];
  for (int d = d0; d < d1; d++) {
    lb[d] = (int64_t)run;
    run += cnt(d);
  }
  __syncthreads();
  // exclusive scans of the two 256-bin histograms by warps 0 and 1 (8 bins per lane)
  if (w < 2) {
    unsigned long long* h = w ? s_hi : s_lo;
    int64_t* out = a.bases + ((size_t)blockIdx.x * 2 + w) * 257;
    unsigned long long v[8], sum = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { v[i] = h[lane * 8 + i]; sum += v[i]; }
    const uint64_t inc = warp_incl_scan(sum);
    uint64_t r = inc - sum;
#pragma unroll
    for (int i = 0; i < 8; i++) { out[lane * 8 + i] = (int64_t)r; r += v[i]; }
    if (lane == 31) out[256] = (int64_t)r;
  }
}

// exchange of one sorted part (see exchange_kernel) that also counts the next pass's full digit per
// (destination GPU, destination part): next_dense[(r*V + v)][d'] += 1
struct ExchVrArgs {
  const Elt* src;
  int64_t m;
  int32_t shift;
  uint32_t mask;
  const int64_t* localbase;
  const int64_t* mybase;
  int64_t per;
  int32_t world;
  Elt* dst[8];
  int32_t has_next, next_shift;
  uint32_t next_mask;
  int32_t V, next_nb;
  int64_t pstart[17];      // first local index of every destination part (the same cut on every GPU); [V] = per
  unsigned* next_dense;    // [G][V][next_nb]
  uint32_t korder;         // key-order flags (ORD instantiations)
};

// EX_THREADS = 512 when the exchange has the SMs to itself or shares them with partition_kernel CTAs that
// come and go; 256 (12.8 K registers) fits beside three resident CTAs of the persistent one-pass kernel.
// EX_U = 16-byte elements in flight per thread.
template <int EX_THREADS, int EX_U, bool ORD>
__global__ void __launch_bounds__(EX_THREADS) exchange_vr_kernel(const ExchVrArgs a) {
  __shared__ Elt* s_dst[8];
  __shared__ long long s_lim[8];
  __shared__ long long s_pstart[17];
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < 8; q++) {
      s_dst[q] = a.dst[q];
      s_lim[q] = (long long)q * a.per;
    }
  }
  if (threadIdx.x < 17) s_pstart[threadIdx.x] = a.pstart[threadIdx.x];
  __syncthreads();
  unsigned pend_slot = 0xffffffffu, pend_cnt = 0;
  const int64_t chunk = (int64_t)EX_THREADS * EX_U;
  const int64_t span = ((a.m + a.world - 1) / a.world + chunk - 1) / chunk * chunk;
  const int64_t chunks_per_span = span / chunk;
  const int64_t total = chunks_per_span * a.world;
  for (int64_t k = blockIdx.x; k < total; k += gridDim.x) {
    const int64_t c0 = (k % a.world) * span + (k / a.world) * chunk;
    if (c0 >= a.m) continue;
    Elt e[EX_U];
#pragma unroll
    for (int u = 0; u < EX_U; u++) {
      const int64_t i = c0 + u * EX_THREADS + threadIdx.x;
      if (i < a.m) e[u] = ld_stream(a.src + i);
    }
#pragma unroll
    for (int u = 0; u < EX_U; u++) {
      const int64_t i = c0 + u * EX_THREADS + threadIdx.x;
      if (i < a.m) {
        const uint64_t dk = digit_key<ORD>(e[u].key, a.korder);
        const unsigned d = (unsigned)(dk >> a.shift) & a.mask;
        const long long g = __ldg(a.mybase + d) + (i - __ldg(a.localbase + d));
        int r = 0;
        for (int q = 1; q < a.world; q++) r += (g >= s_lim[q]);
        const long long j = g - s_lim[r];
        st_elt(s_dst[r] + j, e[u]);
        if (a.has_next) {
          int v = 0;
          for (int q = 1; q < a.V; q++) v += (j >= s_pstart[q]);
          const unsigned dn = (unsigned)(dk >> a.next_shift) & a.next_mask;
          const unsigned slot = (unsigned)(r * a.V + v) * (unsigned)a.next_nb + dn;
          // skew: when the whole warp counts into one slot, one lane adds the population count; a thread also
          // holds back a run of equal slots and adds it once (constant digits: one atomic per thread per launch)
          const unsigned act = __activemask();
          const int leader = __ffs(act) - 1;
          const bool same = __all_sync(act, slot == __shfl_sync(act, slot, leader));
          const unsigned cnt = same ? (((int)(threadIdx.x & 31) == leader) ? (unsigned)__popc(act) : 0u) : 1u;
          if (cnt) {
            if (slot == pend_slot) pend_cnt += cnt;
            else {
              if (pend_cnt) atomicAdd(a.next_dense + pend_slot, pend_cnt);
              pend_slot = slot;
              pend_cnt = cnt;
            }
          }
        }
      }
    }
  }
  if (pend_cnt) atomicAdd(a.next_dense + pend_slot, pend_cnt);
}

// How many distinct values does digit (shift, mask) take over the first `m` (<= 65 536) elements?  The exchange
// kernel's fused next-digit count uses one L2 atomic per element, which is only cheap when the digit has thousands
// of live bins; the host reads this estimate (minimum over the GPUs) to decide per pass.
template <bool ORD>
__global__ void __launch_bounds__(1024) live_bins_kernel(const Elt* src, int m, int shift, uint32_t mask, unsigned* out,
                                                         uint32_t korder) {
  __shared__ unsigned bits[2048];  // 65 536-bit bitmap
  __shared__ unsigned total;
  for (int i = threadIdx.x; i < 2048; i += 1024) bits[i] = 0;
  if (threadIdx.x == 0) total = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < m; i += 1024) {
    const unsigned d = (unsigned)(digit_key<ORD>(ld_stream_key(src + i), korder) >> shift) & mask;
    atomicOr(&bits[d >> 5], 1u << (d & 31));
  }
  __syncthreads();
  unsigned c = 0;
  for (int i = threadIdx.x; i < 2048; i += 1024) c += __popc(bits[i]);
  atomicAdd(&total, c);
  __syncthreads();
  if (threadIdx.x == 0) *out = total;
}

// ------------------------------------------------------------------------------------
// verification: strictly increasing (key,val) + multiset hash (mpi/mpi_lsbsort.cpp:710-739)
// ------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t k, uint64_t v) {
  uint64_t x = k * 0x9E3779B97F4A7C15ULL + (v ^ 0xD6E8FEB86659FD93ULL);
  x ^= x >> 32; x *= 0xD6E8FEB86659FD93ULL;
  x ^= x >> 29; x *= 0x9E3779B97F4A7C15ULL;
  x ^= x >> 32;
  return x;
}

// out[0..3] = checksum of the raw records (sum mix, xor mix, xor key, sum val); out[4] = order violations of
// (digit_key(key), val)
template <bool ORD>
__global__ void __launch_bounds__(256) verify_kernel(const Elt* src, int64_t m, unsigned long long* out, uint32_t korder) {
  uint64_t s = 0, x = 0, xk = 0, sv = 0, bad = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    const Elt e = ld_stream(src + i);
    const uint64_t h = mix64(e.key, e.val);
    s += h; x ^= h; xk ^= e.key; sv += e.val;
    if (i > 0) {
      const Elt p = ld_stream(src + i - 1);
      const uint64_t pk = digit_key<ORD>(p.key, korder), ek = digit_key<ORD>(e.key, korder);
      if (pk > ek || (pk == ek && p.val >= e.val)) bad++;
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, d);
    x ^= __shfl_xor_sync(0xffffffffu, x, d);
    xk ^= __shfl_xor_sync(0xffffffffu, xk, d);
    sv += __shfl_xor_sync(0xffffffffu, sv, d);
    bad += __shfl_xor_sync(0xffffffffu, bad, d);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out + 0, (unsigned long long)s);
    atomicXor(out + 1, (unsigned long long)x);
    atomicXor(out + 2, (unsigned long long)xk);
    atomicAdd(out + 3, (unsigned long long)sv);
    if (bad) atomicAdd(out + 4, (unsigned long long)bad);
  }
}

}  // namespace lsb
