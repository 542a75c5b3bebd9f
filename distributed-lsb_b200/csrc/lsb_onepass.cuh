// lsb_onepass.cuh -- one reference pass (a stable scatter on a digit of 9..16 bits,
// mpi/mpi_lsbsort.cpp:213-247 called once per pass at :494) as ONE persistent sm_100a kernel
// that moves every element through HBM once: 16 B read + 16 B written per element per pass.
//
// Why it is not a plain 65 536-way scatter: a tile of a few thousand elements holds about as
// many distinct 16-bit digits as elements, so neither coalesced stores nor per-tile offsets
// (decoupled look-back over 65 536 bins) are possible from one tile.  The pass is therefore run
// on SUPERTILES of ~650 Ki elements that live in the 126 MB L2 between two steps:
//
//   K1(s)  tile t of supertile s: bulk-load the tile from HBM (cp.async.bulk, evict-first), rank
//          it by the LOW byte of the digit (ballot ranking), write it back sorted by low byte to
//          the supertile scratch X[s % NX] (contiguous, L2 evict-last) and publish, per low byte,
//          {offset, count} of its piece.  No cross-tile dependency at all.
//   K2(s)  segment `lo` of supertile s = all its elements whose low byte is `lo`: gather the
//          T1 pieces (one per K1 tile, in tile order == input order) out of L2 with one small
//          bulk copy each, rank by the HIGH byte, and store every element straight to its final
//          place dst[F[hi][lo] + rank]: F is the running frontier of the 65 536 output bins,
//          advanced once per (supertile, segment) -- supertiles are taken in input order, so
//          the scatter is stable, i.e. exactly `B[starts[bucket]++] = A[i]` (:241-246).
//          A segment larger than a tile (skewed keys) is cut into sub-tiles that run in parallel
//          and find their offsets by decoupled look-back over the 256 high-byte bins.
//
// One persistent CTA grid (4 CTAs of 256 threads per SM) runs both steps: work items are tickets
// from ONE counter, in the order K1(0) .. K1(lead) K2(0) K1(lead+1) K2(1) ...; every dependency
// points to a smaller ticket and every claimed ticket is held by a running CTA, so spinning on
// flags cannot deadlock (a watchdog turns a would-be hang into an error).  HBM sees one read of the
// input and one write of the output as long as the scratch stays in L2 (measured: up to ~40 MB of
// it does; DESIGN.md section 3 has the numbers and why the two-step shape is still the default).
//
// This file also holds digit_hist_kernel: the counts of digits of up to 16 bits (65 536 packed
// shared-memory counters per CTA) that the pass needs up front and that the multi-GPU pass uses per part.
#pragma once
#include "lsb_kernels.cuh"

namespace lsb {

// ------------------------------------------------------------------------------------
// small PTX helpers
// ------------------------------------------------------------------------------------
// (l2_policy and bulk_load_hint live in lsb_kernels.cuh, next to bulk_load)
__device__ __forceinline__ void st_elt_hint(Elt* p, const Elt& e, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.v2.u64 [%0], {%1, %2}, %3;" ::"l"(p), "l"(e.key), "l"(e.val), "l"(policy)
               : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u32(unsigned* p, unsigned v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ------------------------------------------------------------------------------------
// the pass kernel
// ------------------------------------------------------------------------------------
constexpr uint64_t OP_ST_AGG = 1ULL << 62;     // look-back word: count of this sub-tile only
constexpr uint64_t OP_ST_PREFIX = 2ULL << 62;  // look-back word: absolute position after this sub-tile
constexpr uint64_t OP_VAL_MASK = (1ULL << 40) - 1;
constexpr uint64_t OP_TAG_MASK = 0x3fffffULL << 40;
constexpr int OP_MAX_T1 = 256;                  // K1 tiles per supertile (one gather thread per piece)

struct OnePassArgs {
  const Elt* src;
  Elt* dst;
  int64_t m;            // elements
  int32_t shift;        // first bit of the digit; low byte = bits [shift, shift+8)
  int32_t hi_bits;      // width of the high part (1..8)
  int32_t T1;           // K1 tiles per (full) supertile
  int32_t NX;           // supertile scratch buffers
  int32_t nsuper;       // supertiles
  int32_t lead;         // K2(s) is claimed after K1(s + lead)
  int32_t hints;        // bit0 src evict_first, bit1 X evict_last, bit2 X gather evict_last, bit3 dst evict_first
  Elt* X;               // [NX][T1 * TILE]
  unsigned* oc;         // [NX][256][T1]: (count << 16) | offset of piece (tile, low byte)
  uint64_t* lookback;   // [NX][T1 + 256][256]
  uint64_t* F;          // [256 low][256 high]: (version << 40) | next output index of the bin; version v
                        // = the word holds the base for supertile v
  // control block, zeroed before every launch
  unsigned* err;        // != 0: a wait timed out (deadlock watchdog), the launch is void
  unsigned* ticket;     // the one claim counter
  unsigned* done1;      // [nsuper]: K1 tiles finished
  unsigned* done2;      // [nsuper]: sub-tiles of K2(s) that no longer need X[s % NX]
  unsigned* free2;      // [nsuper]: 1 once X[s % NX] may be overwritten (every gather of K2(s) is done)
  unsigned* ready2;     // [nsuper]: 1 | (nbig << 8) once the schedule of K2(s) is published
  unsigned* limit2;     // [nsuper]: number of sub-tiles of K2(s)
  unsigned* totals;     // [nsuper][256]: elements of segment lo of supertile s
  unsigned* segrow;     // [nsuper][256]: exclusive prefix of sub-tiles per segment (look-back ring row)
  unsigned* subclaim;   // [nsuper][256]: next sub-tile of a segment that has more than one
  unsigned* biglist;    // [nsuper][256]: the segments with more than one sub-tile
  unsigned long long timeout_ns;
  unsigned long long* prof;  // [OP_NPROF] stage clocks (LSB_OP_PROF builds only)
  uint32_t korder;      // key-order flags (ORD instantiations)
};

// wait until *p >= want; false on time-out or when another CTA already gave up
__device__ __noinline__ bool op_wait_ge(const unsigned* p, unsigned want, const OnePassArgs& a) {
  unsigned long long t0 = 0;
  for (unsigned n = 1;; n++) {
    if (ld_acquire_u32(p) >= want) return true;
    __nanosleep(32);
    if ((n & 255u) == 0) {
      if (ld_relaxed_u32(a.err)) return false;
      const unsigned long long now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > a.timeout_ns) {
        atomicExch(a.err, 1u);
        return false;
      }
    }
  }
}

// LSB_OP_PROF build (tools/ only): thread 0 of every CTA accumulates clock64() deltas per stage of
// an item and adds them to a.prof[] on exit; the product build compiles none of it.
#ifdef LSB_OP_PROF
#define OP_T(i)                                   \
  do {                                            \
    if (threadIdx.x == 0) {                       \
      const long long now_ = clock64();           \
      prof_acc[i] += now_ - prof_t;               \
      prof_t = now_;                              \
    }                                             \
  } while (0)
#else
#define OP_T(i) do {} while (0)
#endif
constexpr int OP_NPROF1 = 24;  // one-pass kernel's own stage clocks
constexpr int OP_NPROF = 40;   // the whole table: 0..23 one-pass kernel, 24..39 partition_kernel (PT_PROF0)

// K1 tile body after the tile has landed in shared memory: rank by the low byte, publish the
// pieces, write the tile sorted by low byte into its place in the supertile scratch.
template <class C, bool FULL, bool BYTE, bool ORD>
__device__ __forceinline__ void k1_tile(const OnePassArgs& a, const Elt* s_raw, unsigned short* s_perm,
                                        unsigned short* s_whist, unsigned* s_wtot, int count, int s, int slot, int idx,
                                        Elt* xo, uint64_t pol_x) {
  const int tid = threadIdx.x;
  unsigned info[C::IPT], info_p;
  const RowPlan rp = FULL ? RowPlan{0, 0, 0} : row_plan<C>(count);
  op_rank<C, FULL, BYTE, ORD>(s_raw, rp, a.shift, 255u, a.korder, s_whist, info, info_p);
  __syncthreads();
  if (tid < 256) {
    unsigned tile_count, binstart;
    op_scan<C>(s_whist, s_wtot, tile_count, binstart);
    st_relaxed_u32(a.oc + ((size_t)(slot * 256 + tid) * a.T1 + idx), (tile_count << 16) | binstart);
    if (tile_count) atomicAdd(a.totals + (size_t)s * 256 + tid, tile_count);
  }
  __syncthreads();
  op_perm<C, FULL>(rp, s_whist, s_perm, info, info_p);
  __syncthreads();
#pragma unroll
  for (int k = 0; k < C::IPT; k++) {
    const int p = k * C::THREADS + tid;
    if (FULL || p < count) st_elt_hint(xo + p, s_raw[s_perm[p]], pol_x);
  }
}

// Work items are tickets from ONE counter.  Ticket t -> step t / (T1 + 256): the first T1 tickets
// of a step are the K1 tiles of supertile `step`, the other 256 are the segments of supertile
// `step - lead`.  Every dependency of an item points to a smaller ticket, every claimed ticket is
// held by a running CTA, so the spin-waits below cannot deadlock.
template <class C, bool BYTE, bool ORD>
__global__ void __launch_bounds__(C::THREADS, C::MINB) onepass_kernel(const OnePassArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  Elt* s_raw = reinterpret_cast<Elt*>(smem + C::SMEM_RAW);
  unsigned short* s_perm = reinterpret_cast<unsigned short*>(smem + C::SMEM_PERM);
  unsigned short* s_whist = reinterpret_cast<unsigned short*>(smem + C::SMEM_WHIST);
  Elt** s_binptr = reinterpret_cast<Elt**>(smem + C::SMEM_BINDST);
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_kind, s_s, s_idx, s_abort, s_j, s_nbig, s_count, s_T1s, s_lastg;
  __shared__ unsigned s_wtot[8];
  __shared__ unsigned s_wsum[C::WARPS];

  constexpr int DISP = 32;  // the dispatcher thread (lane 0 of warp 1); warp 0 completes K1 tiles
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t S = (int64_t)a.T1 * C::TILE;
  const int ring_rows = a.T1 + 256;
  const uint64_t pol_src = l2_policy((a.hints & 1) ? 1 : 0);
  const uint64_t pol_x = l2_policy((a.hints & 2) ? 2 : 0);
  const uint64_t pol_gather = l2_policy((a.hints & 4) ? 2 : 0);
  const uint64_t pol_dst = l2_policy((a.hints & 8) ? 1 : 0);
  const int shift_hi = a.shift + 8;
  const unsigned mask_hi = (1u << a.hi_bits) - 1u;
  const unsigned period = (unsigned)a.T1 + 256u;
  const unsigned total_tickets = (unsigned)(a.nsuper + a.lead) * period;

  if (tid == 0) {
    mbar_init(&s_bar, 1);
    s_abort = 0;
  }
  unsigned parity = 0;
  unsigned next_t = 0;  // dispatcher: the ticket claimed in advance
  if (tid == DISP) next_t = atomicAdd(a.ticket, 1u);
  __syncthreads();
#ifdef LSB_OP_PROF
  long long prof_acc[OP_NPROF1];
  for (int i = 0; i < OP_NPROF1; i++) prof_acc[i] = 0;
  long long prof_t = clock64();
#endif

  // number of K1 tiles of supertile s (the last one may be short)
  auto tiles1 = [&](int s) -> int {
    const int64_t left = a.m - (int64_t)s * S;
    return (int)(((left < S ? left : S) + C::TILE - 1) / C::TILE);
  };

  while (true) {
    // ------------------------------ dispatch ------------------------------
    if (tid == DISP) {
      int kind = -1, s = 0, idx = 0;
      unsigned t = next_t;
      while (t < total_tickets) {  // skip the tickets of absent items (short last supertile, lead-in)
        const int step = (int)(t / period), r = (int)(t % period);
        if (r < a.T1) {
          if (step < a.nsuper && r < tiles1(step)) { kind = 0; s = step; idx = r; break; }
        } else if (step >= a.lead) {
          kind = 1; s = step - a.lead; idx = r - a.T1; break;
        }
        t = atomicAdd(a.ticket, 1u);
      }
      if (kind >= 0) next_t = atomicAdd(a.ticket, 1u);  // in flight while this item is processed
      bool ok = true;
      if (kind == 0) {
        // X[slot] and oc[slot] were last used by supertile s - NX: all its sub-tiles must have
        // finished gathering before this tile overwrites them
        if (s >= a.NX) ok = op_wait_ge(a.free2 + (s - a.NX), 1u, a);
        const int64_t begin = (int64_t)s * S + (int64_t)idx * C::TILE;
        const int64_t left = a.m - begin;
        const unsigned cnt = (unsigned)(left < C::TILE ? left : C::TILE);
        s_count = (int)cnt;
        if (ok) {
          fence_proxy_async();
          mbar_expect_tx(&s_bar, cnt * 16u);
          bulk_load_hint(s_raw, a.src + begin, cnt * 16u, &s_bar, pol_src);
        }
      } else if (kind == 1) {
        ok = op_wait_ge(a.ready2 + s, 1u, a);  // every K1 tile of supertile s is in X
        s_nbig = (int)(ld_relaxed_u32(a.ready2 + s) >> 8);
      }
      if (!ok) s_abort = 1;
      s_kind = kind;
      s_s = s;
      s_idx = idx;
      s_T1s = kind >= 0 ? tiles1(s) : 0;
    }
    for (int i = tid; i < C::WARPS * 128; i += C::THREADS) reinterpret_cast<unsigned*>(s_whist)[i] = 0;
    __syncthreads();
    if (s_abort) break;
    const int kind = s_kind, s = s_s, idx = s_idx;
    if (kind < 0) break;
    const int slot = s % a.NX;
    const int T1s = s_T1s;
    OP_T(1);  // dispatch

    if (kind == 0) {
      // =============================== K1: tile `idx` of supertile s ===============================
      const int count = s_count;
      mbar_wait(&s_bar, parity);
      parity ^= 1u;
      OP_T(3);  // K1: tile load
      Elt* xo = a.X + (size_t)slot * S + (size_t)idx * C::TILE;
      if (count == C::TILE) k1_tile<C, true, BYTE, ORD>(a, s_raw, s_perm, s_whist, s_wtot, count, s, slot, idx, xo, pol_x);
      else k1_tile<C, false, BYTE, ORD>(a, s_raw, s_perm, s_whist, s_wtot, count, s, slot, idx, xo, pol_x);
      __syncthreads();
      OP_T(7);  // K1: rank, scan, write
      // completion by warp 0 while the dispatcher already prepares the next item: the tile's X
      // stores become visible (fence) before the tile counts as done; whoever finishes the last
      // tile of the supertile publishes the schedule of K2(s)
      if (warp == 0) {
        unsigned old = 0;
        if (lane == 0) {
          __threadfence();
          old = atomicAdd(a.done1 + s, 1u);
        }
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old == (unsigned)T1s - 1u) {
          __threadfence();
          // sub-tiles per segment (at least one, so that every segment's frontier version
          // advances), their exclusive prefix = look-back ring rows, the segments with several
          unsigned ns[8], sum = 0, nb = 0;
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const unsigned tot = ld_relaxed_u32(a.totals + (size_t)s * 256 + lane * 8 + i);
            ns[i] = tot ? (tot + C::TILE - 1) / C::TILE : 1u;
            sum += ns[i];
            nb += ns[i] > 1;
          }
          unsigned incl = sum, bincl = nb;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
            const unsigned ob = __shfl_up_sync(0xffffffffu, bincl, d);
            if (lane >= d) { incl += o; bincl += ob; }
          }
          unsigned row = incl - sum, bi = bincl - nb;
#pragma unroll
          for (int i = 0; i < 8; i++) {
            st_relaxed_u32(a.segrow + (size_t)s * 256 + lane * 8 + i, row);
            row += ns[i];
            if (ns[i] > 1) st_relaxed_u32(a.biglist + (size_t)s * 256 + bi++, (unsigned)(lane * 8 + i));
          }
          const unsigned all = __shfl_sync(0xffffffffu, incl, 31), allbig = __shfl_sync(0xffffffffu, bincl, 31);
          if (lane == 31) st_relaxed_u32(a.limit2 + s, all);
          __syncwarp();
          if (lane == 0) {
            __threadfence();
            st_release_u32(a.ready2 + s, 1u | (allbig << 8));
          }
        }
      }
      OP_T(8);  // K1: completion
    } else {
      // ================ K2: segment `idx` of supertile s, then help with the big segments ================
      const int nbig = s_nbig;
      for (int h = -1; h < nbig; h++) {
        int lo = idx;
        if (h >= 0) {
          lo = (int)ld_relaxed_u32(a.biglist + (size_t)s * 256 + h);
          if (lo == idx) continue;  // my own segment: already exhausted
        }
        const int tot = (int)ld_relaxed_u32(a.totals + (size_t)s * 256 + lo);
        const int row0 = (int)ld_relaxed_u32(a.segrow + (size_t)s * 256 + lo);
        const int ns = tot ? (tot + C::TILE - 1) / C::TILE : 1;
        for (bool first = true;; first = false) {
          int j = 0;
          if (ns == 1) {
            if (!first) break;
          } else {  // several CTAs may work on this segment: sub-tiles are claimed one by one
            __syncthreads();
            if (tid == DISP) s_j = (int)atomicAdd(a.subclaim + (size_t)s * 256 + lo, 1u);
            __syncthreads();
            j = s_j;
            if (j >= ns) break;
            if (!first || h >= 0)
              for (int i = tid; i < C::WARPS * 128; i += C::THREADS) reinterpret_cast<unsigned*>(s_whist)[i] = 0;
          }
          // ---- sub-tile j of segment lo: elements [j * TILE, ...) of the segment ----
          const int sub_begin = j * C::TILE;
          const int count = min(C::TILE, tot - sub_begin);
          const bool last = sub_begin + count >= tot;
          // piece (tile t, this segment): count and offset inside the tile's sorted copy in X
          unsigned pc = 0, poff = 0;
          if (tid < T1s) {
            const unsigned v = ld_relaxed_u32(a.oc + ((size_t)(slot * 256 + lo) * a.T1 + tid));
            pc = v >> 16;
            poff = v & 0xffffu;
          }
          unsigned incl = pc;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const unsigned o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
          }
          if (lane == 31) s_wsum[warp] = incl;
          if (tid == 0 && count > 0) {
            fence_proxy_async();
            mbar_expect_tx(&s_bar, (unsigned)count * 16u);
          }
          __syncthreads();
          OP_T(11);  // K2: piece table + scan
          if (pc) {  // gather: one bulk copy (TMA engine, L2 -> shared) per piece
            int pbeg = (int)(incl - pc);
            for (int i = 0; i < warp; i++) pbeg += (int)s_wsum[i];
            const int cb = max(pbeg, sub_begin), ce = min(pbeg + (int)pc, sub_begin + count);
            if (cb < ce)
              bulk_load_hint(s_raw + (cb - sub_begin), a.X + (size_t)slot * S + (size_t)tid * C::TILE + poff + (cb - pbeg),
                             (unsigned)(ce - cb) * 16u, &s_bar, pol_gather);
          }
          if (count > 0) {
            mbar_wait(&s_bar, parity);
            parity ^= 1u;
          }
          OP_T(12);  // K2: gather
          // X[slot] is no longer needed by this sub-tile; the last one of the supertile releases the slot
          if (tid == 0) s_lastg = atomicAdd(a.done2 + s, 1u) + 1u == ld_relaxed_u32(a.limit2 + s);

          unsigned info[C::IPT], info_p;
          const RowPlan rp = row_plan<C>(count);
          op_rank<C, false, BYTE, ORD>(s_raw, rp, shift_hi, mask_hi, a.korder, s_whist, info, info_p);
          __syncthreads();
          OP_T(13);  // K2: rank
          if (s_lastg && tid == 0) st_release_u32(a.free2 + s, 1u);
          if (tid < 256) {
            unsigned tile_count, binstart;
            op_scan<C>(s_whist, s_wtot, tile_count, binstart);
            // where this sub-tile's elements of bin `tid` start in dst: sub-tile 0 takes it from the
            // frontier word once it carries this supertile's version; later sub-tiles by decoupled
            // look-back over the earlier sub-tiles of the segment
            uint64_t* fw = a.F + lo * 256 + tid;
            uint64_t* my_word = a.lookback + ((size_t)(slot * ring_rows + row0 + j) * 256 + tid);
            const uint64_t tag = ((uint64_t)(s + 1) << 40) & OP_TAG_MASK;
            if (j > 0) st_relaxed_gpu(my_word, OP_ST_AGG | tag | (uint64_t)tile_count);
            uint64_t base = 0;
            int look = j - 1;
            unsigned long long t0 = 0;
            for (unsigned spins = 1;; spins++) {
              if (j == 0) {
                const uint64_t v = ld_relaxed_gpu(fw);
                if ((v >> 40) == (uint64_t)s) { base = v & OP_VAL_MASK; break; }
              } else {
                const uint64_t v = ld_relaxed_gpu(my_word - (size_t)(j - look) * 256);
                if ((v & OP_TAG_MASK) == tag && (v >> 62) != 0) {
                  base += v & OP_VAL_MASK;
                  if ((v >> 62) == 2) break;
                  look--;
                  continue;
                }
              }
              __nanosleep(20);
              if ((spins & 1023u) == 0) {
                const unsigned long long now = globaltimer_ns();
                if (t0 == 0) t0 = now;
                else if (now - t0 > a.timeout_ns || ld_relaxed_u32(a.err)) {
                  atomicExch(a.err, 2u);
                  s_abort = 1;
                  break;
                }
              }
            }
            const uint64_t incl_abs = base + tile_count;
            if (!last) st_relaxed_gpu(my_word, OP_ST_PREFIX | tag | incl_abs);
            else st_relaxed_gpu(fw, ((uint64_t)(s + 1) << 40) | incl_abs);
            s_binptr[tid] = a.dst + ((long long)base - (long long)binstart);
          }
          __syncthreads();
          if (s_abort) break;
          OP_T(14);  // K2: scan + frontier
          op_perm<C, false>(rp, s_whist, s_perm, info, info_p);
          __syncthreads();
          OP_T(15);  // K2: permutation
#pragma unroll
          for (int k = 0; k < C::IPT; k++) {
            const int p = k * C::THREADS + tid;
            if (p < count) {
              const Elt el = s_raw[s_perm[p]];
              st_elt_hint(s_binptr[(unsigned)(digit_key<ORD>(el.key, a.korder) >> shift_hi) & mask_hi] + p, el, pol_dst);
            }
          }
          OP_T(20);  // K2: scatter
        }
        if (s_abort) break;
      }
      if (s_abort) break;
      __syncthreads();  // every thread is done with this item's shared memory
    }
  }
#ifdef LSB_OP_PROF
  if (tid == 0 && a.prof) {
    for (int i = 0; i < OP_NPROF1 - 1; i++) atomicAdd(a.prof + i, (unsigned long long)prof_acc[i]);
    atomicAdd(a.prof + OP_NPROF1 - 1, 1ULL);
  }
#endif
}

// F[lo][hi] = starts[(hi << 8) | lo] + add: the frontier table of a pass from the exclusive scan of
// its digit counts (natural digit order, as global_scan_kernel / part_prep_kernel write it)
__global__ void __launch_bounds__(256) onepass_prep_kernel(const int64_t* starts, int nb, long long add, uint64_t* F) {
  const int i = blockIdx.x * 256 + threadIdx.x;  // i = lo * 256 + hi
  if (i >= 65536) return;
  const int lo = i >> 8, hi = i & 255;
  const int d = (hi << 8) | lo;
  F[i] = d < nb ? (uint64_t)((long long)starts[d] + add) : 0;  // version 0
}

// ------------------------------------------------------------------------------------
// digit counts (localShuffle's count loop, mpi/mpi_lsbsort.cpp:226-229) for digits of up to 16
// bits: one CTA per SM keeps up to 65 536 packed 16-bit counters (128 KiB) in shared memory and
// flushes them once.  Bit 15 of a counter is a guard: the increment that sets it moves 0x8000
// to the global table and clears it again, so a counter can never carry into its neighbour.
// A CTA counts the digits of ONE role (a subset of the sort's digits whose tables fit 128 KiB);
// the `nroles` CTAs of a group read the same keys (HBM once, the others hit L2).
// ------------------------------------------------------------------------------------
constexpr int DH_THREADS = 1024;
constexpr int DH_MAX_DIGITS = 16;
constexpr int DH_SMEM = 65536 * 2;

struct DigitHistArgs {
  const Elt* src;
  int64_t m;
  int32_t nroles;
  int32_t role_first[5];              // digits [role_first[r], role_first[r+1]) belong to role r
  int32_t shift[DH_MAX_DIGITS];
  uint32_t mask[DH_MAX_DIGITS];
  int32_t smem_off[DH_MAX_DIGITS];    // first counter of the digit in the CTA's table
  int32_t out_off[DH_MAX_DIGITS];     // first bin of the digit in `out`
  void* out;                          // u64 or u32 bins, caller zeroes
  int32_t out_u32;
  uint32_t korder;                    // key-order flags (ORD instantiations)
};

__device__ __forceinline__ void dh_global_add(const DigitHistArgs& a, int bin, unsigned v) {
  if (a.out_u32) atomicAdd(reinterpret_cast<unsigned*>(a.out) + bin, v);
  else atomicAdd(reinterpret_cast<unsigned long long*>(a.out) + bin, (unsigned long long)v);
}

// add `c` (1..32) to packed counter `idx`
__device__ __forceinline__ void dh_add(unsigned* sh, int idx, unsigned c, const DigitHistArgs& a, int gbin) {
  const unsigned sft = (idx & 1) * 16;
  const unsigned old = atomicAdd(sh + (idx >> 1), c << sft);
  const unsigned f = (old >> sft) & 0xffffu;
  if (!(f & 0x8000u) && ((f + c) & 0x8000u)) {  // this add set the guard bit
    atomicSub(sh + (idx >> 1), 0x8000u << sft);
    dh_global_add(a, gbin, 0x8000u);
  }
}

template <int NDIG, bool ORD>  // digits per role (0 = run-time count)
__global__ void __launch_bounds__(DH_THREADS, 1) digit_hist_kernel(const DigitHistArgs a) {
  extern __shared__ __align__(16) unsigned dh_sh[];
  const int role = blockIdx.x % a.nroles;
  const int group = blockIdx.x / a.nroles, ngroups = gridDim.x / a.nroles;
  if (group >= ngroups) return;
  const int d0 = a.role_first[role], d1 = NDIG ? d0 + NDIG : a.role_first[role + 1];
  for (int i = threadIdx.x; i < DH_SMEM / 16; i += DH_THREADS) reinterpret_cast<uint4*>(dh_sh)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  constexpr int U = 8;
  const int64_t chunk = (int64_t)DH_THREADS * U;
  const int64_t nchunks = (a.m + chunk - 1) / chunk;
  for (int64_t c = group; c < nchunks; c += ngroups) {
    const int64_t base = c * chunk + threadIdx.x;
    uint64_t k[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int64_t i = base + (int64_t)u * DH_THREADS;
      ok[u] = i < a.m;
      k[u] = ok[u] ? ld_stream_key(a.src + i) : 0;
    }
    // after all U loads: an encode inside the conditional load above makes each load wait for the previous one
#pragma unroll
    for (int u = 0; u < U; u++) k[u] = digit_key<ORD>(k[u], a.korder);
    const bool whole = base - threadIdx.x + chunk <= a.m;  // CTA-uniform: no lane is out of range
#pragma unroll
    for (int u = 0; u < U; u++) {
      for (int d = d0; d < d1; d++) {
        const unsigned bin = (unsigned)(k[u] >> a.shift[d]) & a.mask[d];
        if (whole) {
          // skew: when the whole warp hits one bin, one lane adds 32 instead of a 32-way
          // same-address atomic
          const bool same = __all_sync(0xffffffffu, bin == __shfl_sync(0xffffffffu, bin, 0));
          if (!same) dh_add(dh_sh, a.smem_off[d] + (int)bin, 1u, a, a.out_off[d] + (int)bin);
          else if ((threadIdx.x & 31) == 0) dh_add(dh_sh, a.smem_off[d] + (int)bin, 32u, a, a.out_off[d] + (int)bin);
        } else if (ok[u]) {
          dh_add(dh_sh, a.smem_off[d] + (int)bin, 1u, a, a.out_off[d] + (int)bin);
        }
      }
    }
  }
  __syncthreads();
  for (int d = d0; d < d1; d++) {
    const int nb = (int)a.mask[d] + 1;
    for (int b = threadIdx.x; b < nb; b += DH_THREADS) {
      const int idx = a.smem_off[d] + b;
      const unsigned v = (dh_sh[idx >> 1] >> ((idx & 1) * 16)) & 0xffffu;
      if (v) dh_global_add(a, a.out_off[d] + b, v);
    }
  }
}

// per digit: is one bin holding every element?  (a stable pass on a constant digit is the
// identity: the host may skip it; flags[p] = 1)
__global__ void __launch_bounds__(256) constant_digit_kernel(const unsigned long long* hist, const int* off, const int* nb,
                                                             unsigned long long here, int* flags) {
  __shared__ int found;
  if (threadIdx.x == 0) found = 0;
  __syncthreads();
  const unsigned long long* h = hist + off[blockIdx.x];
  for (int b = threadIdx.x; b < nb[blockIdx.x]; b += 256)
    if (h[b] == here) found = 1;
  __syncthreads();
  if (threadIdx.x == 0) flags[blockIdx.x] = found;
}

}  // namespace lsb
