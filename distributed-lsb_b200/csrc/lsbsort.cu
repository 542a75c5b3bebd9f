// lsbsort.cu -- C ABI (include/lsbsort.h) over the sm_100a kernels in lsb_kernels.cuh /
// lsb_onepass.cuh.
//
// Host-side restatement of the reference's pass structure, mpi/mpi_lsbsort.cpp:481-585
// (globalShuffle / mySort), for device-resident shards.
//
//   G == 1 : ONE read of the shard counts every (sub-)digit of the sort; then, per reference pass,
//            default: two stable 8-bit counting-sort steps over HBM (low bits, then high bits --
//              the same permutation as one stable step on the full digit), partition_kernel;
//            LSB_FLAG_ONE_PASS: ONE launch that moves every element through HBM once
//              (onepass_kernel, lsb_onepass.cuh) for digits of 9..16 bits.
//   G  > 1 : the shard is cut into V parts (virtual ranks g*V+q).  Counts of the full digit per
//            part are known before the pass starts (first pass: counted; later: produced by the
//            previous pass's exchange kernel), NCCL reduce-scatter/all-gather + digit-major /
//            rank-minor exclusive scan (== :327-479) give every part its global offsets, then per
//            part: one local stable sort by the digit (same kernels as G == 1, == localShuffle,
//            :213-247) into a scratch, and an exchange kernel that stores every run straight into
//            the owning GPU's other shard over NVLink (== :530-576) while the next part is being
//            sorted.
//
// Which shape is the default is a measured choice (DESIGN.md section 6): on one B200 both take
// ~15.5 ms per 16-bit pass of 2^30 elements (the one-pass kernel is bound by its instruction
// stream and barrier skew, the two steps by HBM), and next to an exchange kernel the one-pass
// kernel's L2-resident scratch is evicted, so the two-step shape is the default.
#include "../../include/lsbsort.h"
#include "lsb_kernels.cuh"
#include "lsb_onepass.cuh"
#include "lsb_io.cuh"
#include "lsb_segments.cuh"
#include "lsb_lexsort.cuh"
#include "lsb_unique.cuh"

#include <nccl.h>  // types only: the library itself is bound at run time, see NcclApi
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace lsb;

namespace {

typedef PartCfg<512, 11, 2> TileCfg;   // 5632-element tiles, 109 KiB, 2 CTAs (32 warps) per SM
typedef PartCfg<256, 11, 4> TileCfgS;  // 2816-element tiles, 56 KiB, 4 CTAs (32 warps) per SM

struct SubPass {
  int shift;
  int bits;
};

struct PassPlan {
  int shift;    // first bit of the digit
  int bits;     // width of the digit (radix_bits, or the remainder for the last pass)
  int lo_bits;  // low sub-digit width (0 if the digit fits one step)
  int hi_bits;
};

// process-wide tunables read by lsb_create (lsb_tune); defaults are what bench.py measures
struct Tuning {
  int op_cfg = 1;        // one-pass tile shape: 0 = 512 threads x 11 (2 CTAs/SM), 1 = 256 x 11 (4 CTAs/SM)
  int op_persist = 0;    // MiB of L2 set aside for persisting (evict_last) lines, 0 = leave the device default
  int op_t1 = 232;       // K1 tiles per supertile of the one-pass kernel (<= 256): segments of ~2550 elements
  int op_nx = 6;         // supertile scratch buffers
  int op_lead = 3;       // K2(s) is claimed after K1(s + lead): ~2 waves of tickets between a tile and its use
  int op_hints = 15;     // L2 eviction hints, see OnePassArgs::hints
  int op_ctas_mgpu = 3;  // one-pass CTAs per SM while an exchange kernel shares the GPU (G > 1)
  int vparts = 16;       // parts per shard of the multi-GPU pass
  int vramp = 130;       // part q+1 is vramp/100 times part q up to the middle of the shard, then shrinks the same
                         // way: a pass is (sort of the first part) + (all exchanges) when the exchange is the
                         // bottleneck and (all sorts) + (exchange of the last part) otherwise; 100 = equal parts
  int ex_ctas = 1;       // exchange CTAs per SM
  int ex_threads = 0;    // threads per exchange CTA (256 or 512; 0 = by pass shape)
  int ex_u = 4;          // 16-byte elements in flight per exchange thread (4 or 8)
  int timeout_ms = 4000; // watchdog of the one-pass kernel's waits
  int pt_direct = 1;     // partition_kernel: tile = blockIdx.x and the load is issued first (0 = tiles from a ticket counter)
  int pt_chunks = 2;     // partition_kernel: log2 of the bulk copies a tile arrives in (a warp waits for its own piece)
  int pt_variant = 1;    // partition_kernel: 1 = L2 prefetch of a later tile (template L2PF), 0 = off
  int pt_pf_tiles = 0;   // L2PF: how many tiles ahead; 0 = half the SM count (74 on a B200 = a quarter of the
                         // resident CTAs, ~3 us ahead of the tile's own CTA).  Measured at 2^30 (7.09 ms per launch
                         // without): 74 or 148 tiles -> 6.48 ms, 296 -> 6.91 ms, 592 -> 7.66 ms (the prefetched
                         // lines do not survive in L2 next to the output stream), profiles/r2_final_sweep.log
};
Tuning g_tune;

}  // namespace

struct lsb_ctx {
  lsb_config cfg;
  Tuning tune;
  int G = 1, my = 0;
  int64_t n = 0, per = 0, here = 0, first = 0, per_stream = 0;
  int npasses = 0;
  cudaStream_t stream = nullptr;
  Elt* buf[2] = {nullptr, nullptr};  // A, B
  int cur = 0;                        // which of buf[] holds the data
  Elt* peer[2][LSB_MAX_GPUS] = {};    // peer[b][g]: shard b of GPU g (own pointer for g == my)
  bool peer_open[2][LSB_MAX_GPUS] = {};
  int num_sms = 0;
  int tile = TileCfg::TILE;           // elements per tile of partition_kernel
  int op_tile = TileCfg::TILE;        // elements per tile of onepass_kernel
  // partition_kernel (two-step shape; digits of <= 8 bits)
  uint64_t* lookback = nullptr;
  size_t lookback_tiles = 0;
  uint32_t* tile_counters = nullptr;  // [TILE_COUNTERS], recycled
  int next_counter = 0;
  int gen = 0;
  int64_t* seg_start = nullptr;       // [1 + V][2]: {0, here}, then {0, m_q} per part
  uint32_t* seg_tiles = nullptr;      // [1 + V][2]: {0, tiles}
  // sub-digit counts of a whole sort, two-step shape (G == 1)
  unsigned long long* hist = nullptr;        // [HIST_MAX_SUB][256]
  int64_t* scan_out = nullptr;               // [HIST_MAX_SUB][257]
  unsigned long long* host_hist = nullptr;   // pinned [HIST_MAX_SUB][256]
  // digit counts of a whole sort (one-pass shape, G == 1) / of one pass
  unsigned long long* hist16 = nullptr;  // [<= 4 * 65536] counts of every pass's digit, compact
  int64_t* starts16 = nullptr;           // their exclusive scans (natural digit order)
  int* dig_meta = nullptr;               // [2][64] device: offset / bins per pass
  int* skip_flags = nullptr;             // [64] device
  int* host_skip = nullptr;              // [64] pinned
  unsigned long long* counts_all = nullptr;    // [G][65536] (lsb_starts without virtual ranks)
  int64_t* mybase = nullptr;                   // [65536]
  // one-pass kernel
  int64_t op_S = 0;                   // elements per supertile
  Elt* op_X = nullptr;                // [NX][S] supertile scratch (stays in L2)
  unsigned* op_oc = nullptr;          // [NX][256][T1]
  unsigned char* op_ctl = nullptr;    // control block + look-back ring, zeroed before every launch
  size_t op_ctl_bytes = 0;
  uint64_t* op_F = nullptr;           // [65536] frontier table
  unsigned* op_err = nullptr;         // watchdog word, zeroed per call
  unsigned long long* op_prof = nullptr;  // stage clocks of LSB_OP_PROF builds
  int op_resident = 0;                // CTAs per SM the kernel can keep resident
  // pipelined pass (virtual ranks): shard cut into V parts
  bool two_level = false;
  int V = 8;
  int64_t pstart[LSB_MAX_PARTS + 1] = {};    // first local index of every part (the same cut on every GPU)
  int64_t vpart_max = 0;                     // elements of the largest part
  Elt* scratch[2] = {nullptr, nullptr};      // part-sized scratch: the sorted part until it is exchanged
  unsigned* dense_local = nullptr;           // [V][65536] counts of the full digit per part (first pass)
  unsigned* next_dense = nullptr;            // [G][V][65536] counted by the exchange kernel for the next pass
  unsigned* dense_mine = nullptr;            // [V][65536] after the reduce-scatter
  unsigned* c_all = nullptr;                 // [G*V][65536] counts of every virtual rank
  unsigned long long* totals = nullptr;      // [65536] scratch of the virtual-rank scan
  int64_t* digit_base = nullptr;             // [65536] scratch of the virtual-rank scan
  int64_t* mybase_v = nullptr;               // [V][65536]
  int64_t* localbase_v = nullptr;            // [V][65536]
  int64_t* bases_v = nullptr;                // [V][2][257]
  int dense_ready_digit = -1;                // digit whose dense counts already sit in c_all
  unsigned* fuse_live = nullptr;             // [64] device: live-bin estimates per pass
  bool fuse_ok[64] = {};                     // pass p's digit may be counted by pass p-1's exchange kernel
  cudaStream_t xstream = nullptr;            // exchange stream (highest priority)
  cudaEvent_t ev_sorted[LSB_MAX_PARTS] = {}, ev_x[LSB_MAX_PARTS] = {};
  std::vector<cudaEvent_t> xev;              // exchange kernel start/stop pairs (LSB_FLAG_PHASE_EVENTS)
  unsigned long long* small = nullptr;       // [64] scratch: sent[8], verify[5], barrier word, gather
  unsigned long long* small_all = nullptr;   // [G][16]
  unsigned long long* host_small = nullptr;  // pinned [8*16 + 64]
  ncclComm_t comm = nullptr;
  bool comm_ready = false;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  cudaEvent_t ev_caller = nullptr;  // lsb_sort_device: the caller's stream up to the call
  std::vector<cudaEvent_t> phase_ev;
  std::vector<int> phase_kind;  // 0 count, 1 scan/collective, 2 scatter (one-pass / partition), 3 exchange
  int64_t launches = 0;
  int64_t part_elems = 0;
  int skipped = 0;
  std::string err;
};

namespace {

constexpr int TILE_COUNTERS = 1024;

thread_local std::string g_create_err;

// NCCL is bound with dlopen on first multi-GPU use instead of at link time: a process that
// also hosts PyTorch must end up with ONE libnccl.so.2 (torch's bundled 2.28 needs symbols the
// system 2.27 lacks), so if one is already loaded we take that, else the loader's default.
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*ReduceScatter)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
  bool load() {
    if (handle) return true;
    handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!handle) handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!handle) { error = std::string("dlopen libnccl.so.2: ") + dlerror(); return false; }
#define LSB_SYM(field, name)                                            \
    *reinterpret_cast<void**>(&field) = dlsym(handle, name);           \
    if (!field) { error = std::string("dlsym ") + name; handle = nullptr; return false; }
    LSB_SYM(GetUniqueId, "ncclGetUniqueId");
    LSB_SYM(CommInitRank, "ncclCommInitRank");
    LSB_SYM(CommDestroy, "ncclCommDestroy");
    LSB_SYM(AllGather, "ncclAllGather");
    LSB_SYM(AllReduce, "ncclAllReduce");
    LSB_SYM(ReduceScatter, "ncclReduceScatter");
    LSB_SYM(GetErrorString, "ncclGetErrorString");
#undef LSB_SYM
    return true;
  }
};
NcclApi g_nccl;

int fail(lsb_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg; else g_create_err = msg;
  return code;
}

#define CU(c, expr)                                                                          \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return fail(c, LSB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));     \
  } while (0)

#define NC(c, expr)                                                                          \
  do {                                                                                       \
    ncclResult_t r_ = (expr);                                                                \
    if (r_ != ncclSuccess)                                                                   \
      return fail(c, LSB_ERR_NCCL, std::string(#expr) + ": " + g_nccl.GetErrorString(r_));  \
  } while (0)

inline int64_t div_ceil(int64_t a, int64_t b) { return (a + b - 1) / b; }

constexpr uint32_t KEY_ORDER_FLAGS = LSB_FLAG_KEY_I64 | LSB_FLAG_KEY_F64 | LSB_FLAG_DESCENDING;

// What one run of passes sorts: the low `bits` bits of the key word, read through order_key(key, korder) when korder
// is not 0 (the ORD = true instantiation of every digit-reading kernel), as the raw uint64 otherwise.  The one-pass
// kernel's residency, taken at lsb_create for the context's instantiation, holds for the other one too: both are
// bounded by the same __launch_bounds__ and dynamic shared memory.
struct KeyPlan {
  int bits;         // 64, or W for a narrow key (the last digit is clamped to it)
  uint32_t korder;  // the context's key-order flags, or 0 when the key word already holds the order key
};

KeyPlan context_plan(const lsb_ctx* c) { return {64, c->cfg.flags & KEY_ORDER_FLAGS}; }

// A narrow key's pack writes its order key into the low W bits of the key word: its passes sort those as a uint64
// ascending.  At radix 13 a 32-bit key is digits of 13, 13 and 6 bits, never 7 raw key bits.
KeyPlan key_type_plan(const lsb_ctx* c, uint32_t key_type) {
  const int bits = key_type_bits(key_type);
  return bits < 64 ? KeyPlan{bits, 0} : context_plan(c);
}

int num_passes(const lsb_ctx* c, const KeyPlan& k) { return (int)div_ceil(k.bits, c->cfg.radix_bits); }

PassPlan plan_pass(const lsb_ctx* c, const KeyPlan& k, int digit) {
  PassPlan p;
  p.shift = c->cfg.radix_bits * digit;
  p.bits = std::min<int>(c->cfg.radix_bits, k.bits - p.shift);
  // one-pass kernel: low BYTE, then the rest; two-step shape: balanced split (longer runs per bin)
  if (p.bits <= 8) p.lo_bits = 0;
  else p.lo_bits = (c->cfg.flags & LSB_FLAG_ONE_PASS) ? 8 : p.bits / 2;
  p.hi_bits = p.bits - p.lo_bits;
  return p;
}

int phase_mark(lsb_ctx* c, int kind) {
  if (!(c->cfg.flags & LSB_FLAG_PHASE_EVENTS)) return LSB_OK;
  cudaEvent_t ev;
  CU(c, cudaEventCreate(&ev));
  CU(c, cudaEventRecord(ev, c->stream));
  c->phase_ev.push_back(ev);
  c->phase_kind.push_back(kind);
  return LSB_OK;
}

int begin_call(lsb_ctx* c) {
  for (auto ev : c->phase_ev) cudaEventDestroy(ev);
  for (auto ev : c->xev) cudaEventDestroy(ev);
  c->phase_ev.clear();
  c->phase_kind.clear();
  c->xev.clear();
  c->launches = 0;
  c->part_elems = 0;
  c->skipped = 0;
  c->next_counter = 0;
  CU(c, cudaMemsetAsync(c->tile_counters, 0, TILE_COUNTERS * sizeof(uint32_t), c->stream));
  CU(c, cudaMemsetAsync(c->op_err, 0, sizeof(unsigned), c->stream));
  CU(c, cudaEventRecord(c->ev_start, c->stream));
  return phase_mark(c, -1);
}

int end_call(lsb_ctx* c, lsb_stats* st, int passes, int subpasses) {
  CU(c, cudaEventRecord(c->ev_stop, c->stream));
  CU(c, cudaMemcpyAsync(c->host_small + 8, c->op_err, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  if (c->G > 1) CU(c, cudaMemcpyAsync(c->host_small, c->small, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  CU(c, cudaGetLastError());
  if (*reinterpret_cast<unsigned*>(c->host_small + 8))
    return fail(c, LSB_ERR_STATE, "one-pass kernel: a wait on another tile timed out (watchdog); the result is void");
  if (!st) return LSB_OK;
  memset(st, 0, sizeof(*st));
  float ms = 0;
  CU(c, cudaEventElapsedTime(&ms, c->ev_start, c->ev_stop));
  st->device_ms = ms;
  st->passes = passes;
  st->subpasses = subpasses;
  st->skipped = c->skipped;
  st->elements = c->here;
  st->kernel_launches = c->launches;
  int sp = 0;
  for (size_t i = 1; i < c->phase_ev.size(); i++) {
    float d = 0;
    CU(c, cudaEventElapsedTime(&d, c->phase_ev[i - 1], c->phase_ev[i]));
    switch (c->phase_kind[i]) {
      case 0: st->hist_ms += d; break;
      case 1: st->scan_ms += d; break;
      case 2:
        st->partition_ms += d;
        if (sp < LSB_MAX_SUBPASSES) st->subpass_ms[sp] = d;
        sp++;
        break;
      default: break;  // 3: the tail of a pipelined pass waiting for its last exchange
    }
  }
  for (size_t i = 0; i + 1 < c->xev.size(); i += 2) {
    float d = 0;
    CU(c, cudaEventElapsedTime(&d, c->xev[i], c->xev[i + 1]));
    st->exchange_ms += d;
  }
  st->partition_launches = subpasses;
  st->partition_elements = c->part_elems;
  if (c->G > 1) {
    for (int g = 0; g < c->G; g++) st->sent[g] = (int64_t)c->host_small[g];
  } else {
    st->sent[0] = c->here;
  }
  return LSB_OK;
}

// ---- kernel launch helpers -----------------------------------------------------------

// counts of `ndig` digits over src[0, m) in ONE read (localShuffle's count loop, :226-229):
// digit i of width bits[i] at shift[i] is accumulated into out[out_off[i] ...] (u64 or u32
// bins, the caller zeroes them).  Digits are packed into at most 4 roles of <= 65 536 bins.
int launch_digit_hist(lsb_ctx* c, uint32_t korder, const Elt* src, int64_t m, const int* shift, const int* bits, const int* out_off,
                      int ndig, void* out, bool out_u32) {
  for (int first = 0; first < ndig;) {
    DigitHistArgs a;
    memset(&a, 0, sizeof(a));
    a.src = src;
    a.m = m;
    a.out = out;
    a.out_u32 = out_u32 ? 1 : 0;
    a.korder = korder;
    int nd = 0, role = 0, role_bins = 0;
    a.role_first[0] = 0;
    while (first + nd < ndig && nd < DH_MAX_DIGITS) {
      const int nb = 1 << bits[first + nd];
      if (role_bins + nb > 65536) {
        if (role == 3) break;
        a.role_first[++role] = nd;
        role_bins = 0;
      }
      a.shift[nd] = shift[first + nd];
      a.mask[nd] = (uint32_t)(nb - 1);
      a.smem_off[nd] = role_bins;
      a.out_off[nd] = out_off[first + nd];
      role_bins += nb;
      nd++;
    }
    a.nroles = role + 1;
    for (int r = a.nroles; r < 5; r++) a.role_first[r] = nd;
    if (m > 0) {
      const int64_t chunks = div_ceil(m, (int64_t)DH_THREADS * 8);
      const int groups = (int)std::max<int64_t>(1, std::min<int64_t>(c->num_sms / a.nroles, chunks));
      bool one_each = true;
      for (int r = 0; r < a.nroles; r++) one_each = one_each && (a.role_first[r + 1] - a.role_first[r] == 1);
      const int grid = groups * a.nroles;
      if (korder) {
        if (one_each) digit_hist_kernel<1, true><<<grid, DH_THREADS, DH_SMEM, c->stream>>>(a);
        else digit_hist_kernel<0, true><<<grid, DH_THREADS, DH_SMEM, c->stream>>>(a);
      } else {
        if (one_each) digit_hist_kernel<1, false><<<grid, DH_THREADS, DH_SMEM, c->stream>>>(a);
        else digit_hist_kernel<0, false><<<grid, DH_THREADS, DH_SMEM, c->stream>>>(a);
      }
      c->launches++;
      CU(c, cudaGetLastError());
    }
    first += nd;
  }
  return LSB_OK;
}

template <bool ORD>
void launch_subdigit_hist_kernel(const HistArgs& a, int grid, bool bytes, cudaStream_t stream) {
#define LSB_HIST(N, B) subdigit_hist_kernel<N, B, ORD><<<grid, HIST_THREADS, 0, stream>>>(a)
  if (bytes && a.nsub == 8) LSB_HIST(8, true);
  else switch (a.nsub) {
    case 1: LSB_HIST(1, false); break;
    case 2: LSB_HIST(2, false); break;
    case 3: LSB_HIST(3, false); break;
    case 4: LSB_HIST(4, false); break;
    case 5: LSB_HIST(5, false); break;
    case 6: LSB_HIST(6, false); break;
    case 7: LSB_HIST(7, false); break;
    case 8: LSB_HIST(8, false); break;
    case 9: LSB_HIST(9, false); break;
    case 10: LSB_HIST(10, false); break;
    case 11: LSB_HIST(11, false); break;
    case 12: LSB_HIST(12, false); break;
    case 13: LSB_HIST(13, false); break;
    case 14: LSB_HIST(14, false); break;
    case 15: LSB_HIST(15, false); break;
    default: LSB_HIST(16, false); break;
  }
#undef LSB_HIST
}

// 256-bin histograms of up to HIST_MAX_SUB sub-digits in one read + their exclusive scans (two-step shape)
int launch_subdigit_hist(lsb_ctx* c, uint32_t korder, const Elt* src, const SubPass* subs, int nsub) {
  CU(c, cudaMemsetAsync(c->hist, 0, sizeof(unsigned long long) * 256 * HIST_MAX_SUB, c->stream));
  if (c->here > 0) {
    HistArgs a;
    memset(&a, 0, sizeof(a));
    a.src = src;
    a.m = c->here;
    a.nsub = nsub;
    for (int s = 0; s < nsub; s++) {
      a.shift[s] = subs[s].shift;
      a.mask[s] = (1u << subs[s].bits) - 1;
    }
    a.out = c->hist;
    a.korder = korder;
    const int grid = (int)std::min<int64_t>((int64_t)c->num_sms * 4, div_ceil(c->here, HIST_THREADS));
    bool bytes = true;  // sub-digits are exactly bytes 0..nsub-1 of the key (radix 8 and 16)
    for (int s = 0; s < nsub; s++) bytes = bytes && subs[s].shift == 8 * s && subs[s].bits == 8;
    if (korder) launch_subdigit_hist_kernel<true>(a, grid, bytes, c->stream);
    else launch_subdigit_hist_kernel<false>(a, grid, bytes, c->stream);
    c->launches++;
  }
  CU(c, cudaGetLastError());
  int rc = phase_mark(c, 0);
  if (rc) return rc;
  scan256_kernel<<<nsub, 256, 0, c->stream>>>(c->hist, c->scan_out);
  c->launches++;
  CU(c, cudaGetLastError());
  return phase_mark(c, 1);
}

// exclusive scan of counts[G][nb] in digit-major, rank-minor order -> out[nb] = this rank's column
int launch_scan(lsb_ctx* c, const unsigned long long* counts, int nb, int G, int my, int64_t* out, unsigned long long* sent) {
  GlobalScanArgs s;
  s.counts = counts;
  s.nb = nb;
  s.G = G;
  s.my = my;
  s.per = sent ? c->per : INT64_MAX / 16;
  s.mybase = out;
  s.sent = sent;
  global_scan_kernel<<<1, 1024, 0, c->stream>>>(s);
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

// one stable counting-sort step on <= 8 bits over src[0, m): the whole pass for digits of <= 8
// bits, half a pass in the two-step shape.  bases[bin] = first output index of the bin.
int launch_partition(lsb_ctx* c, uint32_t korder, const Elt* src, int64_t m, int shift, int bits, const int64_t* seg_start,
                     const uint32_t* seg_tile_start, const int64_t* bases, Elt* dst) {
  if (c->gen > 126) {  // tags exhausted: wipe the look-back words and start over
    CU(c, cudaMemsetAsync(c->lookback, 0, c->lookback_tiles * 256 * sizeof(uint64_t), c->stream));
    c->gen = 0;
  }
  if (c->next_counter >= TILE_COUNTERS) {  // stream order: every earlier launch is done with its counter
    CU(c, cudaMemsetAsync(c->tile_counters, 0, TILE_COUNTERS * sizeof(uint32_t), c->stream));
    c->next_counter = 0;
  }
  PartArgs a;
  memset(&a, 0, sizeof(a));
  a.src = src;
  a.shift = shift;
  a.mask = (1u << bits) - 1;
  a.seg_bits = 0;                    // one segment {0, m}: the whole input
  a.seg_start = seg_start;
  a.seg_tile_start = seg_tile_start;
  a.bases = bases;
  a.lookback = c->lookback;
  a.tile_counter = c->tile_counters + c->next_counter++;
  a.tag_agg = (uint64_t)(2 * c->gen + 1) << 56;
  a.tag_inc = (uint64_t)(2 * c->gen + 2) << 56;
  c->gen++;
  a.per = INT64_MAX / 16;
  a.world = 1;
  a.dst[0] = dst;
  a.prof = c->op_prof;
  a.direct = c->tune.pt_direct;
  a.log_chunks = c->tune.pt_chunks;
  a.d_begin = 0;
  a.d_end = m;
  a.pf_tiles = c->tune.pt_pf_tiles > 0 ? c->tune.pt_pf_tiles : std::max(1, c->num_sms / 2);
  a.korder = korder;
  c->part_elems += m;
  if (m > 0) {
    const unsigned grid = (unsigned)div_ceil(m, c->tile);
    const bool l2pf = a.direct && c->tune.pt_variant;  // the prefetch needs blockIdx-ordered tiles
    if (korder) {
      if (l2pf) partition_kernel<TileCfg, true, true><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
      else partition_kernel<TileCfg, false, true><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
    } else {
      if (l2pf) partition_kernel<TileCfg, true, false><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
      else partition_kernel<TileCfg, false, false><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
    }
    c->launches++;
  }
  CU(c, cudaGetLastError());
  return phase_mark(c, 2);
}

// one stable scatter on a digit of 9..16 bits over src[0, m) -> dst: starts[d] + add is the first
// output index of digit d (natural digit order); `ctas_per_sm` 0 = as many as stay resident
int launch_onepass(lsb_ctx* c, uint32_t korder, const Elt* src, Elt* dst, int64_t m, int shift, int bits, const int64_t* starts,
                   long long add, int ctas_per_sm) {
  c->part_elems += m;
  if (m > 0) {
    const int T1 = c->tune.op_t1, NX = c->tune.op_nx;
    const int nsuper = (int)div_ceil(m, c->op_S);
    // control block layout for this launch (u32 words), then the look-back ring (u64)
    size_t w = 0;
    auto take = [&](size_t n) { size_t o = w; w += n; return o; };
    const size_t o_ticket = take(4), o_done1 = take(nsuper), o_done2 = take(nsuper), o_free2 = take(nsuper), o_ready2 = take(nsuper),
                 o_limit2 = take(nsuper), o_totals = take(256 * (size_t)nsuper), o_segrow = take(256 * (size_t)nsuper),
                 o_subclaim = take(256 * (size_t)nsuper), o_biglist = take(256 * (size_t)nsuper);
    w = (w + 3) & ~(size_t)3;
    const size_t ring_bytes = (size_t)NX * (T1 + 256) * 256 * sizeof(uint64_t);
    const size_t bytes = w * 4 + ring_bytes;
    if (bytes > c->op_ctl_bytes) return fail(c, LSB_ERR_STATE, "one-pass control block too small");
    CU(c, cudaMemsetAsync(c->op_ctl, 0, bytes, c->stream));
    onepass_prep_kernel<<<256, 256, 0, c->stream>>>(starts, 1 << bits, add, c->op_F);
    OnePassArgs a;
    memset(&a, 0, sizeof(a));
    a.src = src;
    a.dst = dst;
    a.m = m;
    a.shift = shift;
    a.hi_bits = bits - 8;
    a.T1 = T1;
    a.NX = NX;
    a.nsuper = nsuper;
    a.lead = c->tune.op_lead;
    a.hints = c->tune.op_hints;
    a.X = c->op_X;
    a.oc = c->op_oc;
    unsigned* ctl = reinterpret_cast<unsigned*>(c->op_ctl);
    a.lookback = reinterpret_cast<uint64_t*>(c->op_ctl + w * 4);
    a.F = c->op_F;
    a.err = c->op_err;
    a.ticket = ctl + o_ticket;
    a.done1 = ctl + o_done1;
    a.done2 = ctl + o_done2;
    a.free2 = ctl + o_free2;
    a.ready2 = ctl + o_ready2;
    a.limit2 = ctl + o_limit2;
    a.totals = ctl + o_totals;
    a.segrow = ctl + o_segrow;
    a.subclaim = ctl + o_subclaim;
    a.biglist = ctl + o_biglist;
    a.timeout_ns = (unsigned long long)c->tune.timeout_ms * 1000000ULL;
    a.prof = c->op_prof;
    a.korder = korder;
    const int per_sm = ctas_per_sm > 0 ? std::min(ctas_per_sm, c->op_resident) : c->op_resident;
    // every claimed item must belong to a resident CTA: never launch more CTAs than fit
    const int64_t useful = div_ceil(m, c->op_tile) + 256;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)c->num_sms * per_sm, useful));
    const bool byte = (shift % 8) == 0 && bits == 16;  // both digit halves are whole bytes of the key
    if (c->tune.op_cfg == 1) {
      if (korder) onepass_kernel<TileCfgS, false, true><<<grid, TileCfgS::THREADS, TileCfgS::SMEM, c->stream>>>(a);
      else if (byte) onepass_kernel<TileCfgS, true, false><<<grid, TileCfgS::THREADS, TileCfgS::SMEM, c->stream>>>(a);
      else onepass_kernel<TileCfgS, false, false><<<grid, TileCfgS::THREADS, TileCfgS::SMEM, c->stream>>>(a);
    } else {
      if (korder) onepass_kernel<TileCfg, false, true><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
      else if (byte) onepass_kernel<TileCfg, true, false><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
      else onepass_kernel<TileCfg, false, false><<<grid, TileCfg::THREADS, TileCfg::SMEM, c->stream>>>(a);
    }
    c->launches += 2;
    CU(c, cudaGetLastError());
  }
  return phase_mark(c, 2);
}

// exchange-free barrier across GPUs, ordered on the sort stream
int stream_barrier(lsb_ctx* c) {
  if (c->G == 1) return LSB_OK;
  NC(c, g_nccl.AllReduce(c->small + 32, c->small + 32, 1, ncclUint64, ncclSum, c->comm, c->stream));
  return LSB_OK;
}

int64_t part_len(const lsb_ctx* c, int q) {
  return std::min<int64_t>(c->pstart[q + 1], c->here) - std::min<int64_t>(c->pstart[q], c->here);
}

// virtual-rank counts of digit `digit` for every part of every GPU -> c_all[G*V][nb]
// (localShuffle's counts, :226-229, per part; then the count exchange of :327-383)
int count_parts(lsb_ctx* c, const KeyPlan& k, int digit) {
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits, V = c->V;
  CU(c, cudaMemsetAsync(c->dense_local, 0, sizeof(unsigned) * (size_t)V * nb, c->stream));
  for (int q = 0; q < V; q++) {
    const int64_t m = part_len(c, q);
    if (m <= 0) continue;
    const int off = q * nb;
    int rc = launch_digit_hist(c, k.korder, c->buf[c->cur] + c->pstart[q], m, &p.shift, &p.bits, &off, 1, c->dense_local, true);
    if (rc) return rc;
  }
  if (c->G > 1) {
    NC(c, g_nccl.AllGather(c->dense_local, c->c_all, (size_t)V * nb, ncclUint32, c->comm, c->stream));
  } else {
    CU(c, cudaMemcpyAsync(c->c_all, c->dense_local, sizeof(unsigned) * (size_t)V * nb, cudaMemcpyDeviceToDevice, c->stream));
  }
  return LSB_OK;
}

// c_all -> mybase_v[q][d] (global output index of part q's first element of digit d: the
// reference's exclusive scan in digit-major / rank-minor order, :327-479, over virtual ranks),
// sent[] (:553-554), localbase_v and the bases of the local step(s) of every part
int part_offsets(lsb_ctx* c, const KeyPlan& k, int digit) {
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits, V = c->V;
  CU(c, cudaMemsetAsync(c->small, 0, 8 * sizeof(unsigned long long), c->stream));
  VrScanArgs v;
  v.counts = c->c_all;
  v.nb = nb;
  v.GV = c->G * V;
  v.first_vr = c->my * V;
  v.V = V;
  v.G = c->G;
  v.per = c->per;
  v.totals = c->totals;
  v.digit_base = c->digit_base;
  v.mybase = c->mybase_v;
  v.sent = c->small;
  vr_totals_kernel<<<(nb + 255) / 256, 256, 0, c->stream>>>(v);
  c->launches++;
  int rc = launch_scan(c, c->totals, nb, 1, 0, c->digit_base, nullptr);
  if (rc) return rc;
  vr_place_kernel<<<(nb + 255) / 256, 256, 0, c->stream>>>(v);
  PartPrepArgs pp;
  pp.counts = c->c_all + (size_t)c->my * V * nb;
  pp.nb = nb;
  pp.lo_bits = p.lo_bits;
  pp.hi_bits = p.hi_bits;
  pp.localbase = c->localbase_v;
  pp.bases = c->bases_v;
  part_prep_kernel<<<V, 1024, 0, c->stream>>>(pp);
  c->launches += 2;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

// c_all (counts of every virtual rank) -> does one digit value hold all n elements?
int digit_is_constant(lsb_ctx* c, const KeyPlan& k, int digit, bool* constant) {
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits;
  VrScanArgs v;
  memset(&v, 0, sizeof(v));
  v.counts = c->c_all;
  v.nb = nb;
  v.GV = c->G * c->V;
  v.totals = c->totals;
  vr_totals_kernel<<<(nb + 255) / 256, 256, 0, c->stream>>>(v);
  const int meta[2] = {0, nb};
  CU(c, cudaMemcpyAsync(c->dig_meta, meta, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(c->dig_meta + 64, meta + 1, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  constant_digit_kernel<<<1, 256, 0, c->stream>>>(c->totals, c->dig_meta, c->dig_meta + 64, (unsigned long long)c->n, c->skip_flags);
  c->launches += 2;
  CU(c, cudaMemcpyAsync(c->host_skip, c->skip_flags, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  *constant = c->host_skip[0] != 0;
  return LSB_OK;
}

// Which passes may have their digit counted by the previous pass's exchange kernel: digits of >= 12 bits that
// take >= 2048 distinct values among the first 65 536 elements of every shard (a digit's distribution does not
// change when the array is permuted, so the input is as good a sample as any).  One host sync, before pass 0.  Every
// digit of the plan is sampled, whichever of its passes the caller runs.
int plan_fusion(lsb_ctx* c, const KeyPlan& k) {
  unsigned* d = c->fuse_live;
  const int m = (int)std::min<int64_t>(c->here, 65536), np = num_passes(c, k);
  for (int p = 0; p < np; p++) {
    const PassPlan q = plan_pass(c, k, p);
    const uint32_t mask = (uint32_t)((1u << q.bits) - 1);
    if (k.korder) live_bins_kernel<true><<<1, 1024, 0, c->stream>>>(c->buf[c->cur], m, q.shift, mask, d + p, k.korder);
    else live_bins_kernel<false><<<1, 1024, 0, c->stream>>>(c->buf[c->cur], m, q.shift, mask, d + p, 0);
    c->launches++;
  }
  CU(c, cudaGetLastError());
  if (c->G > 1) NC(c, g_nccl.AllReduce(d, d, (size_t)np, ncclUint32, ncclMin, c->comm, c->stream));
  CU(c, cudaMemcpyAsync(c->host_skip, d, sizeof(unsigned) * np, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  for (int p = 0; p < np; p++) c->fuse_ok[p] = plan_pass(c, k, p).bits >= 12 && c->host_skip[p] >= 2048;
  return LSB_OK;
}

// one reference pass, pipelined over V parts of the shard (virtual ranks g*V+q):
//   counts of the full digit of every part are known up front (first pass: counted here; later
//   passes: produced by the previous pass's exchange kernel), so
//     part q:   local stable sort by the digit (compute stream)  ->  exchange (exchange stream)
//   and the exchange of part q overlaps the local sort of part q+1.
int pass_global(lsb_ctx* c, const KeyPlan& k, int digit, int* subpasses, bool fuse_next) {
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits;
  const int V = c->V;
  int rc;
  if (c->dense_ready_digit != digit) {  // nobody has counted this digit yet
    if ((rc = count_parts(c, k, digit))) return rc;
    if ((rc = phase_mark(c, 0))) return rc;
  }
  c->dense_ready_digit = -1;
  if (!(c->cfg.flags & LSB_FLAG_NO_SKIP) && c->n > 0) {
    // a digit that is constant over the WHOLE array makes the pass the identity (every GPU sees the same
    // counts of all virtual ranks, so every GPU takes the same decision)
    bool constant = false;
    if ((rc = digit_is_constant(c, k, digit, &constant))) return rc;
    if (constant) {  // identity pass: every element stays where it is (sendCounts: everything to myself)
      c->skipped++;
      unsigned long long* sent = c->host_small + 140;
      for (int g = 0; g < 8; g++) sent[g] = (g == c->my) ? (unsigned long long)c->here : 0ULL;
      CU(c, cudaMemcpyAsync(c->small, sent, 8 * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
      return phase_mark(c, 1);
    }
  }
  if ((rc = part_offsets(c, k, digit))) return rc;
  if ((rc = phase_mark(c, 1))) return rc;

  // The exchange kernel counts the NEXT pass's digit per (destination GPU, destination part) with one L2 atomic per
  // element -- cheap when the digit has thousands of bins (lanes of a warp rarely collide), ruinous for narrow digits
  // (radix 8: 256 bins, every warp instruction replays ~32 times: 131 ms per pass measured).  Narrow digits are
  // counted by the shared-memory count kernel at the start of their own pass instead (one extra 16 B/element read).
  int next_nb = 0, next_shift = 0;
  // ... and wide digits that are narrow in THIS data (skewed keys), judged from a sample at the start of the sort
  const bool has_next = fuse_next && digit + 1 < num_passes(c, k) && c->fuse_ok[digit + 1];
  if (has_next) {
    const PassPlan q = plan_pass(c, k, digit + 1);
    next_nb = 1 << q.bits;
    next_shift = q.shift;
    CU(c, cudaMemsetAsync(c->next_dense, 0, sizeof(unsigned) * (size_t)c->G * V * next_nb, c->stream));
  }
  const bool two_step = p.lo_bits && !(c->cfg.flags & LSB_FLAG_ONE_PASS);
  const bool timed = (c->cfg.flags & LSB_FLAG_PHASE_EVENTS) != 0;
  const int xbuf = c->cur ^ 1;
  int last_x = -1, prev_x = -1, sorted_parts = 0;
  for (int q = 0; q < V; q++) {
    const int64_t m = part_len(c, q);
    if (m <= 0) continue;
    const int slot = sorted_parts++ & 1;  // empty parts take no scratch: alternate over the parts that are sorted
    Elt* part = c->buf[c->cur] + c->pstart[q];
    const int64_t* segs = c->seg_start + 2 * (1 + q);
    const uint32_t* tiles = c->seg_tiles + 2 * (1 + q);
    const Elt* sorted;
    if (two_step) {  // low step into the scratch, high step back in place
      if ((rc = launch_partition(c, k.korder, part, m, p.shift, p.lo_bits, segs, tiles, c->bases_v + ((size_t)q * 2 + 0) * 257, c->scratch[0])))
        return rc;
      if ((rc = launch_partition(c, k.korder, c->scratch[0], m, p.shift + p.lo_bits, p.hi_bits, segs, tiles,
                                 c->bases_v + ((size_t)q * 2 + 1) * 257, part)))
        return rc;
      sorted = part;
      (*subpasses) += 2;
    } else {  // one launch; its output lives in an alternating scratch until it has been exchanged
      Elt* out = c->scratch[slot];
      if (prev_x >= 0) CU(c, cudaStreamWaitEvent(c->stream, c->ev_x[prev_x], 0));  // scratch[slot] was read by that exchange
      if (p.lo_bits) rc = launch_onepass(c, k.korder, part, out, m, p.shift, p.bits, c->localbase_v + (size_t)q * nb, 0, c->tune.op_ctas_mgpu);
      else rc = launch_partition(c, k.korder, part, m, p.shift, p.hi_bits, segs, tiles, c->bases_v + ((size_t)q * 2 + 1) * 257, out);
      if (rc) return rc;
      sorted = out;
      (*subpasses)++;
    }
    CU(c, cudaEventRecord(c->ev_sorted[q], c->stream));
    CU(c, cudaStreamWaitEvent(c->xstream, c->ev_sorted[q], 0));
    if (timed) {
      cudaEvent_t e0;
      CU(c, cudaEventCreate(&e0));
      CU(c, cudaEventRecord(e0, c->xstream));
      c->xev.push_back(e0);
    }
    ExchVrArgs x;
    memset(&x, 0, sizeof(x));
    x.src = sorted;
    x.m = m;
    x.shift = p.shift;
    x.mask = (uint32_t)(nb - 1);
    x.localbase = c->localbase_v + (size_t)q * nb;
    x.mybase = c->mybase_v + (size_t)q * nb;
    x.per = c->per;
    x.world = c->G;
    for (int g = 0; g < c->G; g++) x.dst[g] = c->peer[xbuf][g];
    x.has_next = has_next;
    x.next_shift = next_shift;
    x.next_mask = (uint32_t)(next_nb - 1);
    x.V = V;
    x.next_nb = next_nb;
    for (int i = 0; i <= LSB_MAX_PARTS; i++) x.pstart[i] = c->pstart[std::min(i, V)];
    x.next_dense = c->next_dense;
    x.korder = k.korder;
    // 512 threads next to partition_kernel CTAs that come and go; 256 fit beside three resident one-pass CTAs
    const int ex_threads = c->tune.ex_threads ? c->tune.ex_threads : ((c->cfg.flags & LSB_FLAG_ONE_PASS) ? 256 : 512);
    const int ex_u = c->tune.ex_u == 8 ? 8 : 4;
    const int grid = (int)std::min<int64_t>((int64_t)c->num_sms * c->tune.ex_ctas, div_ceil(m, (int64_t)ex_threads * ex_u));
    if (k.korder) {
      if (ex_threads == 256) exchange_vr_kernel<256, 4, true><<<grid, 256, 0, c->xstream>>>(x);
      else if (ex_u == 8) exchange_vr_kernel<512, 8, true><<<grid, 512, 0, c->xstream>>>(x);
      else exchange_vr_kernel<512, 4, true><<<grid, 512, 0, c->xstream>>>(x);
    } else {
      if (ex_threads == 256) exchange_vr_kernel<256, 4, false><<<grid, 256, 0, c->xstream>>>(x);
      else if (ex_u == 8) exchange_vr_kernel<512, 8, false><<<grid, 512, 0, c->xstream>>>(x);
      else exchange_vr_kernel<512, 4, false><<<grid, 512, 0, c->xstream>>>(x);
    }
    c->launches++;
    CU(c, cudaGetLastError());
    if (timed) {
      cudaEvent_t e1;
      CU(c, cudaEventCreate(&e1));
      CU(c, cudaEventRecord(e1, c->xstream));
      c->xev.push_back(e1);
    }
    CU(c, cudaEventRecord(c->ev_x[q], c->xstream));
    prev_x = last_x;
    last_x = q;
  }
  if (last_x >= 0) CU(c, cudaStreamWaitEvent(c->stream, c->ev_x[last_x], 0));
  if ((rc = phase_mark(c, 3))) return rc;
  if (has_next) {
    // sum the G contributions to each of my parts, then share every virtual rank's counts: the two
    // collectives are also the barrier "all peers' stores into my shard have landed"
    if (c->G > 1) {
      NC(c, g_nccl.ReduceScatter(c->next_dense, c->dense_mine, (size_t)V * next_nb, ncclUint32, ncclSum, c->comm, c->stream));
      NC(c, g_nccl.AllGather(c->dense_mine, c->c_all, (size_t)V * next_nb, ncclUint32, c->comm, c->stream));
    } else {
      CU(c, cudaMemcpyAsync(c->c_all, c->next_dense, sizeof(unsigned) * (size_t)V * next_nb, cudaMemcpyDeviceToDevice, c->stream));
    }
    c->dense_ready_digit = digit + 1;
    if ((rc = phase_mark(c, 1))) return rc;
  } else if ((rc = stream_barrier(c))) {
    return rc;
  }
  c->cur = xbuf;
  return LSB_OK;
}

// passes [d0, d1) on one GPU: one read counts the digits of every pass, then one launch per pass
// (LSB_FLAG_ONE_PASS) or per 8-bit step (default) that reads the shard once and writes it once
int passes_single(lsb_ctx* c, const KeyPlan& k, int d0, int d1, int* subpasses) {
  if (!(c->cfg.flags & LSB_FLAG_ONE_PASS)) {
    // two-step shape: one histogram read for all sub-digits, then one HBM -> HBM step per sub-digit
    std::vector<SubPass> subs;
    for (int d = d0; d < d1; d++) {
      const PassPlan p = plan_pass(c, k, d);
      if (p.lo_bits) subs.push_back({p.shift, p.lo_bits});
      subs.push_back({p.shift + p.lo_bits, p.hi_bits});
    }
    int rc;
    for (size_t s0 = 0; s0 < subs.size(); s0 += HIST_MAX_SUB) {
      const int ns = (int)std::min<size_t>(HIST_MAX_SUB, subs.size() - s0);
      if ((rc = launch_subdigit_hist(c, k.korder, c->buf[c->cur], subs.data() + s0, ns))) return rc;
      const bool may_skip = !(c->cfg.flags & LSB_FLAG_NO_SKIP) && c->here > 0;
      if (may_skip) {  // a digit that is constant over the shard makes its stable step the identity
        CU(c, cudaMemcpyAsync(c->host_hist, c->hist, sizeof(unsigned long long) * 256 * ns, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));  // once per sort (per 16 sub-digits), before the first step
      }
      for (int s = 0; s < ns; s++) {
        const SubPass& sp = subs[s0 + s];
        if (may_skip) {
          bool constant = false;
          for (int b = 0; b < 256; b++) constant = constant || c->host_hist[s * 256 + b] == (unsigned long long)c->here;
          if (constant) { c->skipped++; continue; }
        }
        if ((rc = launch_partition(c, k.korder, c->buf[c->cur], c->here, sp.shift, sp.bits, c->seg_start, c->seg_tiles, c->scan_out + (size_t)s * 257, c->buf[c->cur ^ 1])))
          return rc;
        c->cur ^= 1;
        (*subpasses)++;
      }
    }
    return LSB_OK;
  }
  const int np = d1 - d0;
  int shift[64], bits[64], off[64], meta[128];
  int total = 0;
  for (int i = 0; i < np; i++) {
    const PassPlan p = plan_pass(c, k, d0 + i);
    shift[i] = p.shift;
    bits[i] = p.bits;
    off[i] = total;
    meta[i] = total;
    meta[64 + i] = 1 << p.bits;
    total += 1 << p.bits;
  }
  int rc;
  CU(c, cudaMemsetAsync(c->hist16, 0, sizeof(unsigned long long) * total, c->stream));
  if ((rc = launch_digit_hist(c, k.korder, c->buf[c->cur], c->here, shift, bits, off, np, c->hist16, false))) return rc;
  if ((rc = phase_mark(c, 0))) return rc;
  for (int i = 0; i < np; i++)
    if ((rc = launch_scan(c, c->hist16 + off[i], 1 << bits[i], 1, 0, c->starts16 + off[i], nullptr))) return rc;
  const bool may_skip = !(c->cfg.flags & LSB_FLAG_NO_SKIP) && c->here > 0;
  if (may_skip) {  // a digit that is constant over the shard makes its stable pass the identity
    CU(c, cudaMemcpyAsync(c->dig_meta, meta, sizeof(meta), cudaMemcpyHostToDevice, c->stream));
    constant_digit_kernel<<<np, 256, 0, c->stream>>>(c->hist16, c->dig_meta, c->dig_meta + 64, (unsigned long long)c->here, c->skip_flags);
    c->launches++;
    CU(c, cudaMemcpyAsync(c->host_skip, c->skip_flags, sizeof(int) * np, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));  // once per sort, before the first pass
  }
  if ((rc = phase_mark(c, 1))) return rc;
  for (int i = 0; i < np; i++) {
    if (may_skip && c->host_skip[i]) { c->skipped++; continue; }
    const PassPlan p = plan_pass(c, k, d0 + i);
    const int64_t* starts = c->starts16 + off[i];
    if (p.lo_bits == 0) {
      rc = launch_partition(c, k.korder, c->buf[c->cur], c->here, p.shift, p.bits, c->seg_start, c->seg_tiles, starts, c->buf[c->cur ^ 1]);
      (*subpasses)++;
    } else {
      rc = launch_onepass(c, k.korder, c->buf[c->cur], c->buf[c->cur ^ 1], c->here, p.shift, p.bits, starts, 0, 0);
      (*subpasses)++;
    }
    if (rc) return rc;
    c->cur ^= 1;
  }
  return LSB_OK;
}

// the passes [d0, d1) of the plan `k` in the context's pass shape
int run_passes(lsb_ctx* c, const KeyPlan& k, int d0, int d1, int* subpasses) {
  c->dense_ready_digit = -1;
  if (!c->two_level) return passes_single(c, k, d0, d1, subpasses);
  int rc = plan_fusion(c, k);
  if (rc) return rc;
  for (int d = d0; d < d1; d++)
    if ((rc = pass_global(c, k, d, subpasses, d + 1 < d1))) return rc;
  return LSB_OK;
}

int check_ready(lsb_ctx* c) {
  if (!c) return LSB_ERR_ARG;
  if (c->G > 1 && !c->comm_ready) return fail(c, LSB_ERR_STATE, "world_size > 1: call lsb_comm_init first");
  return LSB_OK;
}

// lsb_sort with the plan `k`: the context's, or a narrow-key call's own for the records it packed
int sort_shard(lsb_ctx* c, const KeyPlan& k, lsb_stats* st) {
  CU(c, cudaSetDevice(c->cfg.device));
  int rc = begin_call(c);
  if (rc) return rc;
  int subpasses = 0;
  const int np = num_passes(c, k);
  if ((rc = run_passes(c, k, 0, np, &subpasses))) return rc;
  return end_call(c, st, np, subpasses);
}

// ---- lsb_sort_device: the caller's arrays <-> the shard's records --------------------------------------------------------

inline bool ranges_overlap(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + b_bytes && y < x + a_bytes;
}

// NULL or device memory of this context's device, aligned to its element width, that is not one of its own shards
int check_device_array(lsb_ctx* c, const char* fn, const void* p, const char* name, int64_t count, int elt_bytes = 8) {
  if (!p) return LSB_OK;
  const std::string where = std::string(fn) + ": " + name;
  if ((uintptr_t)p & (elt_bytes - 1)) return fail(c, LSB_ERR_ARG, where + " is not " + std::to_string(elt_bytes) + "-byte aligned");
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();  // not sticky: clear it so that the next launch check does not report it
    return fail(c, LSB_ERR_ARG, where + " is not CUDA memory");
  }
  if (at.type != cudaMemoryTypeDevice || at.device != c->cfg.device)
    return fail(c, LSB_ERR_ARG, where + " is not device memory of device " + std::to_string(c->cfg.device));
  const size_t shard_bytes = (size_t)std::max<int64_t>(c->per, 1) * sizeof(Elt);
  for (int b = 0; b < 2; b++)
    if (ranges_overlap(p, (size_t)count * elt_bytes, c->buf[b], shard_bytes))
      return fail(c, LSB_ERR_ARG, where + " overlaps the context's own shards");
  return LSB_OK;
}

int io_grid(const lsb_ctx* c, int64_t count) {
  return (int)std::min<int64_t>((int64_t)c->num_sms * IO_CTAS_PER_SM, div_ceil(count, IO_THREADS));
}

// expands LSB_KT_CALL(KT) for the key type `key_type` (checked by the caller: LSB_KEY_CONTEXT .. LSB_KEY_BF16)
#define LSB_KT_SWITCH(key_type)                   \
  switch (key_type) {                             \
    case LSB_KEY_U32: LSB_KT_CALL(LSB_KEY_U32); break; \
    case LSB_KEY_I32: LSB_KT_CALL(LSB_KEY_I32); break; \
    case LSB_KEY_F32: LSB_KT_CALL(LSB_KEY_F32); break; \
    case LSB_KEY_U16: LSB_KT_CALL(LSB_KEY_U16); break; \
    case LSB_KEY_I16: LSB_KT_CALL(LSB_KEY_I16); break; \
    case LSB_KEY_F16: LSB_KT_CALL(LSB_KEY_F16); break; \
    case LSB_KEY_BF16: LSB_KT_CALL(LSB_KEY_BF16); break; \
    default: LSB_KT_CALL(LSB_KEY_CONTEXT); break;      \
  }

// flags: the key order of the call (a narrow key's DESCENDING goes into its key word)
int launch_pack(lsb_ctx* c, uint32_t key_type, const void* keys, const uint64_t* vals, uint32_t flags) {
  const PackArgs a{keys, vals, c->buf[0], c->here, c->first, flags};
  const int grid = io_grid(c, c->here);
#define LSB_KT_CALL(KT)                                                    \
  if (vals) pack_kernel<KT, true><<<grid, IO_THREADS, 0, c->stream>>>(a); \
  else pack_kernel<KT, false><<<grid, IO_THREADS, 0, c->stream>>>(a)
  LSB_KT_SWITCH(key_type)
#undef LSB_KT_CALL
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

template <int KBYTES>
void launch_unpack_kernel(const UnpackArgs& a, int grid, cudaStream_t stream) {
  if (a.keys && a.vals) unpack_kernel<KBYTES, true, true><<<grid, IO_THREADS, 0, stream>>>(a);
  else if (a.keys) unpack_kernel<KBYTES, true, false><<<grid, IO_THREADS, 0, stream>>>(a);
  else unpack_kernel<KBYTES, false, true><<<grid, IO_THREADS, 0, stream>>>(a);
}

int launch_unpack(lsb_ctx* c, int key_bytes, void* keys, uint64_t* vals) {
  const UnpackArgs a{c->buf[c->cur], keys, vals, c->here};
  const int grid = io_grid(c, c->here);
  if (key_bytes == 8) launch_unpack_kernel<8>(a, grid, c->stream);
  else if (key_bytes == 4) launch_unpack_kernel<4>(a, grid, c->stream);
  else launch_unpack_kernel<2>(a, grid, c->stream);
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

// ---- lsb_sort_segments_device: offsets check, pack with segment ids, retag, unpack (lsb_segments.cuh) -------------------

// offsets[0] == 0, offsets[nseg] == count, non-decreasing: one flag read back (host_small[16], from small[60])
int segsort_check(lsb_ctx* c, const int64_t* offsets, int64_t nseg, int64_t count, bool* ok) {
  int* bad = reinterpret_cast<int*>(c->small + 60);
  CU(c, cudaMemsetAsync(bad, 0, sizeof(int), c->stream));
  const SegsortCheckArgs a{offsets, nseg, count, bad};
  segsort_check_kernel<<<io_grid(c, nseg), IO_THREADS, 0, c->stream>>>(a);
  c->launches++;
  CU(c, cudaGetLastError());
  CU(c, cudaMemcpyAsync(c->host_small + 16, bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  *ok = *reinterpret_cast<const int*>(c->host_small + 16) == 0;
  return LSB_OK;
}

int launch_segsort_pack(lsb_ctx* c, uint32_t key_type, const void* keys, const int64_t* offsets, int64_t nseg, int idxbits,
                        uint32_t flags) {
  const SegsortPackArgs a{keys, offsets, c->buf[0], c->here, nseg, idxbits, flags};
  const int grid = io_grid(c, c->here);
#define LSB_KT_CALL(KT) segsort_pack_kernel<KT><<<grid, IO_THREADS, 0, c->stream>>>(a)
  LSB_KT_SWITCH(key_type)
#undef LSB_KT_CALL
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

int launch_segsort_retag(lsb_ctx* c, int idxbits, int segw) {
  const SegsortRetagArgs a{c->buf[c->cur], c->here, idxbits, segw};
  segsort_retag_kernel<<<io_grid(c, c->here), IO_THREADS, 0, c->stream>>>(a);
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

template <int KBYTES>
void launch_segsort_unpack_kernel(const SegsortUnpackArgs& a, int grid, int mode, cudaStream_t stream) {
#define LSB_SEG_UNPACK(K, V) segsort_unpack_kernel<KBYTES, K, V><<<grid, IO_THREADS, 0, stream>>>(a)
  const bool keys = a.keys != nullptr;
  switch (mode) {
    case SEGSORT_VALS_NONE: LSB_SEG_UNPACK(true, SEGSORT_VALS_NONE); break;
    case SEGSORT_VALS_GATHER: if (keys) LSB_SEG_UNPACK(true, SEGSORT_VALS_GATHER); else LSB_SEG_UNPACK(false, SEGSORT_VALS_GATHER); break;
    case SEGSORT_VALS_LOCAL: if (keys) LSB_SEG_UNPACK(true, SEGSORT_VALS_LOCAL); else LSB_SEG_UNPACK(false, SEGSORT_VALS_LOCAL); break;
    default: if (keys) LSB_SEG_UNPACK(true, SEGSORT_VALS_GLOBAL); else LSB_SEG_UNPACK(false, SEGSORT_VALS_GLOBAL); break;
  }
#undef LSB_SEG_UNPACK
}

int launch_segsort_unpack(lsb_ctx* c, int key_bytes, void* keys, uint64_t* vals, const uint64_t* vals_in,
                          const int64_t* offsets, bool local, int segw) {
  const SegsortUnpackArgs a{c->buf[c->cur], keys, vals, vals_in, offsets, c->here, segw};
  const int grid = io_grid(c, c->here);
  const int mode = !vals ? SEGSORT_VALS_NONE : vals_in ? SEGSORT_VALS_GATHER : local ? SEGSORT_VALS_LOCAL : SEGSORT_VALS_GLOBAL;
  if (key_bytes == 8) launch_segsort_unpack_kernel<8>(a, grid, mode, c->stream);
  else if (key_bytes == 4) launch_segsort_unpack_kernel<4>(a, grid, mode, c->stream);
  else launch_segsort_unpack_kernel<2>(a, grid, mode, c->stream);
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

// The checks of the two device entry points, in the order they make them: first the context, the key type and the
// count (on success *key_bytes is the key width in bytes) ...
int check_call(lsb_ctx* c, const char* fn, uint32_t key_type, int64_t count, int* key_bytes) {
  int rc = check_ready(c);
  if (rc) return rc;
  const int bits = key_type_bits(key_type);
  if (!bits) return fail(c, LSB_ERR_ARG, std::string(fn) + ": unknown key_type " + std::to_string(key_type));
  if (bits < 64 && (c->cfg.flags & (LSB_FLAG_KEY_I64 | LSB_FLAG_KEY_F64)))
    return fail(c, LSB_ERR_ARG, std::string(fn) + ": a narrow key_type needs a context without LSB_FLAG_KEY_I64 / LSB_FLAG_KEY_F64");
  if (count != c->here) return fail(c, LSB_ERR_ARG, std::string(fn) + ": count must equal this shard's size");
  *key_bytes = bits / 8;
  return LSB_OK;
}

// ... then, for count > 0 and a non-NULL keys_in, the four arrays: an output at least, each of them NULL or device memory
// that check_device_array accepts at its own width
int check_arrays(lsb_ctx* c, const char* fn, int key_bytes, int64_t count, const void* keys_in, const uint64_t* vals_in,
                 const void* keys_out, const uint64_t* vals_out) {
  if (!keys_out && !vals_out) return fail(c, LSB_ERR_ARG, std::string(fn) + ": keys_out and vals_out are both NULL");
  const void* ptrs[4] = {keys_in, vals_in, keys_out, vals_out};
  const char* names[4] = {"keys_in", "vals_in", "keys_out", "vals_out"};
  const int widths[4] = {key_bytes, 8, key_bytes, 8};
  for (int i = 0; i < 4; i++) {
    const int rc = check_device_array(c, fn, ptrs[i], names[i], count, widths[i]);
    if (rc) return rc;
  }
  return LSB_OK;
}

int sort_device(lsb_ctx* c, const char* fn, uint32_t key_type, const void* keys_in, const uint64_t* vals_in, void* keys_out,
                uint64_t* vals_out, int64_t count, void* stream, lsb_stats* st) {
  int kb = 8;
  int rc = check_call(c, fn, key_type, count, &kb);
  if (rc) return rc;
  CU(c, cudaSetDevice(c->cfg.device));
  if (count) {
    if (!keys_in) return fail(c, LSB_ERR_ARG, std::string(fn) + ": keys_in is NULL");
    if ((rc = check_arrays(c, fn, kb, count, keys_in, vals_in, keys_out, vals_out))) return rc;
    if (keys_out && vals_out && ranges_overlap(keys_out, (size_t)count * kb, vals_out, (size_t)count * sizeof(uint64_t)))
      return fail(c, LSB_ERR_ARG, std::string(fn) + ": keys_out and vals_out overlap");
  }
  CU(c, cudaEventRecord(c->ev_caller, (cudaStream_t)stream));
  CU(c, cudaStreamWaitEvent(c->stream, c->ev_caller, 0));
  c->cur = 0;
  if (count && (rc = launch_pack(c, key_type, keys_in, vals_in, c->cfg.flags))) return rc;
  if ((rc = sort_shard(c, key_type_plan(c, key_type), st))) return rc;
  if (count && (rc = launch_unpack(c, kb, keys_out, vals_out))) return rc;
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int sort_segments_device(lsb_ctx* c, const char* fn, uint32_t key_type, const void* keys_in, const uint64_t* vals_in,
                         void* keys_out, uint64_t* vals_out, int64_t count, const int64_t* seg_offsets, int64_t num_segments,
                         uint32_t seg_flags, void* stream, lsb_stats* st) {
  if (!c) return LSB_ERR_ARG;
  if (c->G > 1) return fail(c, LSB_ERR_ARG, std::string(fn) + ": one GPU only (world_size > 1)");
  int kb = 8;
  int rc = check_call(c, fn, key_type, count, &kb);
  if (rc) return rc;
  if (num_segments < 1) return fail(c, LSB_ERR_ARG, std::string(fn) + ": num_segments must be >= 1");
  if (seg_flags & ~LSB_SEG_LOCAL_INDEX) return fail(c, LSB_ERR_ARG, std::string(fn) + ": unknown seg_flags");
  const SegsortLayout lay = segsort_layout(count, num_segments, c->cfg.radix_bits);
  if (!lay.fits)
    return fail(c, LSB_ERR_ARG, std::string(fn) + ": segment id and input index need " + std::to_string(lay.segw + lay.idxbits) +
                                    " bits of one key word (> 64)");
  CU(c, cudaSetDevice(c->cfg.device));
  const size_t bytes = (size_t)count * sizeof(uint64_t), kbytes = (size_t)count * kb;
  const size_t off_bytes = (size_t)(num_segments + 1) * sizeof(int64_t);
  if (count) {
    if (!keys_in || !seg_offsets) return fail(c, LSB_ERR_ARG, std::string(fn) + ": keys_in or seg_offsets is NULL");
    if ((rc = check_arrays(c, fn, kb, count, keys_in, vals_in, keys_out, vals_out))) return rc;
    if ((rc = check_device_array(c, fn, seg_offsets, "seg_offsets", num_segments + 1))) return rc;
    // keys_in is consumed by the pack, so keys_out may alias it; vals_in and the offsets are read by the unpack
    const void* outs[2] = {keys_out, vals_out};
    const char* names[2] = {"keys_out", "vals_out"};
    const size_t out_bytes[2] = {kbytes, bytes};
    for (int i = 0; i < 2; i++) {
      if (!outs[i]) continue;
      if ((i == 0 && vals_out && ranges_overlap(keys_out, kbytes, vals_out, bytes)) ||
          (vals_in && ranges_overlap(outs[i], out_bytes[i], vals_in, bytes)) || ranges_overlap(outs[i], out_bytes[i], seg_offsets, off_bytes))
        return fail(c, LSB_ERR_ARG, std::string(fn) + ": " + names[i] + " overlaps another output, vals_in or seg_offsets");
    }
  }
  CU(c, cudaEventRecord(c->ev_caller, (cudaStream_t)stream));
  CU(c, cudaStreamWaitEvent(c->stream, c->ev_caller, 0));
  if ((rc = begin_call(c))) return rc;
  if (count) {
    bool ok = false;
    if ((rc = segsort_check(c, seg_offsets, num_segments, count, &ok))) return rc;
    if (!ok) return fail(c, LSB_ERR_ARG, std::string(fn) + ": seg_offsets must rise from 0 to count (offsets[0] == 0, "
                                           "offsets[num_segments] == count, non-decreasing)");
  }
  c->cur = 0;
  if (count) {  // one segment: lsb_sort_device's records, {key word, vals_in or the index}
    rc = lay.segbits ? launch_segsort_pack(c, key_type, keys_in, seg_offsets, num_segments, lay.idxbits, c->cfg.flags)
                     : launch_pack(c, key_type, keys_in, vals_in, c->cfg.flags);
    if (rc) return rc;
  }
  const KeyPlan keys = key_type_plan(c, key_type);
  const int key_passes = num_passes(c, keys);
  int subpasses = 0;
  if ((rc = run_passes(c, keys, 0, key_passes, &subpasses))) return rc;
  if (lay.segbits) {
    if (count && (rc = launch_segsort_retag(c, lay.idxbits, lay.segw))) return rc;
    // the segment passes sort the low digits of the retagged key word as a uint64, ascending
    if ((rc = run_passes(c, KeyPlan{64, 0}, 0, lay.passes, &subpasses))) return rc;
  }
  if (count) {
    rc = lay.segbits ? launch_segsort_unpack(c, kb, keys_out, vals_out, vals_in, seg_offsets, seg_flags & LSB_SEG_LOCAL_INDEX, lay.segw)
                     : launch_unpack(c, kb, keys_out, vals_out);
    if (rc) return rc;
  }
  return end_call(c, st, key_passes + lay.passes, subpasses);
}

// ---- lsb_lexsort_device: a round's pack, its passes, ..., the unpack (lsb_lexsort.cuh) ----------------------------------

// the pack of round `r` of `cols`: into buf[0] for the first round, in place on buf[cur] for every later one
// the columns of round `r` with their shifts in the round's word
void round_columns(const lsb_key_column* cols, const LexsortRound& r, LexsortColumn* out) {
  int shift = 0;
  for (int i = 0; i < r.ncols; i++) {
    const lsb_key_column& k = cols[r.first + i];
    out[i] = LexsortColumn{k.keys, k.key_type, k.flags, shift};
    shift += key_type_bits(k.key_type);
  }
}

int launch_lexsort_pack(lsb_ctx* c, const lsb_key_column* cols, const LexsortRound& r, bool gather) {
  LexsortPackArgs a{};
  round_columns(cols, r, a.col);
  a.buf = c->buf[gather ? c->cur : 0];
  a.count = c->here;
  const int grid = io_grid(c, c->here);
#define LSB_LEX_PACK(N)                                                          \
  if (gather) lexsort_pack_kernel<true, N><<<grid, IO_THREADS, 0, c->stream>>>(a); \
  else lexsort_pack_kernel<false, N><<<grid, IO_THREADS, 0, c->stream>>>(a)
  switch (r.ncols) {  // 1 .. LEXSORT_ROUND_COLUMNS (lexsort_rounds)
    case 1: LSB_LEX_PACK(1); break;
    case 2: LSB_LEX_PACK(2); break;
    case 3: LSB_LEX_PACK(3); break;
    default: LSB_LEX_PACK(4); break;
  }
#undef LSB_LEX_PACK
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

int launch_lexsort_unpack(lsb_ctx* c, const uint64_t* vals_in, uint64_t* vals_out) {
  if (!vals_in) return launch_unpack(c, 8, nullptr, vals_out);  // the input index in the val word
  const LexsortUnpackArgs a{c->buf[c->cur], vals_in, vals_out, c->here};
  lexsort_unpack_kernel<<<io_grid(c, c->here), IO_THREADS, 0, c->stream>>>(a);
  c->launches++;
  CU(c, cudaGetLastError());
  return LSB_OK;
}

// The checks of lsb_lexsort_device's context, columns and count, shared by lsb_unique_device: widths[i] is the bit
// width of column i.  Sets the context's device.
int check_columns(lsb_ctx* c, const char* fn, const lsb_key_column* cols, int32_t K, int64_t count, std::vector<int>& widths) {
  const std::string f(fn);
  if (c->G > 1) return fail(c, LSB_ERR_ARG, f + ": one GPU only (world_size > 1)");
  if (c->cfg.flags & KEY_ORDER_FLAGS)
    return fail(c, LSB_ERR_ARG, f + ": the context has key-order flags (KEY_I64 / KEY_F64 / DESCENDING); the columns "
                                    "carry their own");
  if (K < 1 || !cols) return fail(c, LSB_ERR_ARG, f + ": needs num_columns >= 1 and a columns array");
  widths.assign(K, 0);
  for (int i = 0; i < K; i++) {
    const std::string col = f + ": column " + std::to_string(i);
    widths[i] = key_type_bits(cols[i].key_type);
    if (!widths[i]) return fail(c, LSB_ERR_ARG, col + ": unknown key_type " + std::to_string(cols[i].key_type));
    const uint32_t allowed = widths[i] == 64 ? KEY_ORDER_FLAGS : LSB_FLAG_DESCENDING;
    const uint32_t both = LSB_FLAG_KEY_I64 | LSB_FLAG_KEY_F64;
    if ((cols[i].flags & ~allowed) || (cols[i].flags & both) == both)
      return fail(c, LSB_ERR_ARG, col + ": flags " + std::to_string(cols[i].flags) + " are not " +
                                      (widths[i] == 64 ? "DESCENDING plus at most one of KEY_I64 / KEY_F64" : "DESCENDING or 0"));
  }
  if (count != c->here) return fail(c, LSB_ERR_ARG, f + ": count must equal this shard's size");
  CU(c, cudaSetDevice(c->cfg.device));
  for (int i = 0; count && i < K; i++) {
    const std::string name = "column " + std::to_string(i);
    if (!cols[i].keys) return fail(c, LSB_ERR_ARG, f + ": " + name + ": keys is NULL");
    int rc = check_device_array(c, fn, cols[i].keys, name.c_str(), count, widths[i] / 8);
    if (rc) return rc;
  }
  return LSB_OK;
}

// The packs and passes of every round, least significant first: afterwards buf[cur] holds {the last round's word, the
// input index} of every record in lexsort order.  passes counts the passes of every round.
int sort_columns(lsb_ctx* c, const lsb_key_column* cols, const std::vector<LexsortRound>& rounds, int* passes, int* subpasses) {
  c->cur = 0;
  for (size_t r = 0; r < rounds.size(); r++) {
    // the round's word holds its order keys: its passes sort the low `bits` bits as a uint64, ascending
    int rc;
    if (c->here && (rc = launch_lexsort_pack(c, cols, rounds[r], r > 0))) return rc;
    if ((rc = run_passes(c, KeyPlan{rounds[r].bits, 0}, 0, rounds[r].passes, subpasses))) return rc;
    *passes += rounds[r].passes;
  }
  return LSB_OK;
}

std::vector<LexsortRound> column_rounds(const lsb_ctx* c, const std::vector<int>& widths) {
  std::vector<LexsortRound> rounds(widths.size());
  rounds.resize(lexsort_rounds(widths.data(), (int)widths.size(), c->cfg.radix_bits, rounds.data()));
  return rounds;
}

int lexsort_device(lsb_ctx* c, const char* fn, const lsb_key_column* cols, int32_t K, const uint64_t* vals_in,
                   uint64_t* vals_out, int64_t count, void* stream, lsb_stats* st) {
  if (!c) return LSB_ERR_ARG;
  const std::string f(fn);
  std::vector<int> widths;
  int rc = check_columns(c, fn, cols, K, count, widths);
  if (rc) return rc;
  const size_t bytes = (size_t)count * sizeof(uint64_t);
  if (count) {
    if (!vals_out) return fail(c, LSB_ERR_ARG, f + ": vals_out is NULL");
    rc = check_device_array(c, fn, vals_in, "vals_in", count);
    if (!rc) rc = check_device_array(c, fn, vals_out, "vals_out", count);
    if (rc) return rc;
    if (vals_in && ranges_overlap(vals_out, bytes, vals_in, bytes)) return fail(c, LSB_ERR_ARG, f + ": vals_out overlaps vals_in");
    for (int i = 0; i < K; i++)
      if (ranges_overlap(vals_out, bytes, cols[i].keys, (size_t)count * (widths[i] / 8)))
        return fail(c, LSB_ERR_ARG, f + ": vals_out overlaps column " + std::to_string(i));
  }
  CU(c, cudaEventRecord(c->ev_caller, (cudaStream_t)stream));
  CU(c, cudaStreamWaitEvent(c->stream, c->ev_caller, 0));
  if ((rc = begin_call(c))) return rc;
  int passes = 0, subpasses = 0;
  if ((rc = sort_columns(c, cols, column_rounds(c, widths), &passes, &subpasses))) return rc;
  if (count && (rc = launch_lexsort_unpack(c, vals_in, vals_out))) return rc;
  return end_call(c, st, passes, subpasses);
}

// ---- lsb_unique_device: lexsort's rounds (sorted mode), head flags, tile counts and their scan, the outputs -------------
// (lsb_unique.cuh)

template <bool SORTED>
void launch_unique_flag_kernel(const UniqueFlagArgs& a, int ncols, int grid, cudaStream_t stream) {
#define LSB_UNIQ_FLAG(N) unique_flag_kernel<SORTED, N><<<grid, IO_THREADS, 0, stream>>>(a)
  switch (ncols) {  // 1 .. LEXSORT_ROUND_COLUMNS
    case 1: LSB_UNIQ_FLAG(1); break;
    case 2: LSB_UNIQ_FLAG(2); break;
    case 3: LSB_UNIQ_FLAG(3); break;
    default: LSB_UNIQ_FLAG(4); break;
  }
#undef LSB_UNIQ_FLAG
}

template <int PHASE>
void launch_unique_tile_kernel(const UniqueTileArgs& a, int ncols, int grid, cudaStream_t stream) {
#define LSB_UNIQ_TILE(N) unique_tile_kernel<PHASE, N><<<grid, UNIQUE_THREADS, 0, stream>>>(a)
  switch (ncols) {  // 0: the sorted records; 1 .. LEXSORT_ROUND_COLUMNS: the last round's columns
    case 0: LSB_UNIQ_TILE(0); break;
    case 1: LSB_UNIQ_TILE(1); break;
    case 2: LSB_UNIQ_TILE(2); break;
    case 3: LSB_UNIQ_TILE(3); break;
    default: LSB_UNIQ_TILE(4); break;
  }
#undef LSB_UNIQ_TILE
}

// count >= 1.  Sorted mode reads buf[cur], the records of sort_columns; both modes keep their scratch in buf[cur ^ 1].
// U goes to small[24] on the device and comes back to host_small[24] before the call's final synchronise.
int launch_unique(lsb_ctx* c, const lsb_key_column* cols, const std::vector<LexsortRound>& rounds, bool sorted,
                  int64_t* index_out, int64_t* inverse_out, int64_t* counts_out) {
  const UniqueScratch s = unique_scratch(c->buf[c->cur ^ 1], c->here);
  int64_t* u = reinterpret_cast<int64_t*>(c->small + 24);
  for (size_t r = 0; r + 1 < rounds.size(); r++) {
    UniqueFlagArgs f{};
    round_columns(cols, rounds[r], f.col);
    f.rec = c->buf[c->cur];
    f.diff = s.diff;
    f.count = c->here;
    f.first = r == 0;
    if (sorted) launch_unique_flag_kernel<true>(f, rounds[r].ncols, io_grid(c, c->here), c->stream);
    else launch_unique_flag_kernel<false>(f, rounds[r].ncols, io_grid(c, c->here), c->stream);
    c->launches++;
    CU(c, cudaGetLastError());
  }
  UniqueTileArgs a{};
  a.rec = c->buf[c->cur];
  if (!sorted) round_columns(cols, rounds.back(), a.col);
  a.diff = rounds.size() > 1 ? s.diff : nullptr;
  a.count = c->here;
  a.totals = s.totals;
  a.bases = s.bases;
  a.index_out = index_out;
  a.inverse_out = inverse_out;
  a.ends = counts_out ? s.ends : nullptr;
  a.num_unique = u;
  const int ncols = sorted ? 0 : rounds.back().ncols;
  launch_unique_tile_kernel<0>(a, ncols, (int)s.tiles, c->stream);
  c->launches++;
  CU(c, cudaGetLastError());
  // one CTA walks all count / UNIQUE_TILE totals, more than the sort's tables it was sized for: 1.0 ms at 2^30, under 1 %
  // of the call (DESIGN.md §4g)
  int rc = launch_scan(c, s.totals, (int)s.tiles, 1, 0, s.bases, nullptr);
  if (rc) return rc;
  launch_unique_tile_kernel<1>(a, ncols, (int)s.tiles, c->stream);
  c->launches++;
  CU(c, cudaGetLastError());
  if (counts_out) {
    const UniqueCountsArgs k{s.ends, u, counts_out, c->here};
    unique_counts_kernel<<<io_grid(c, c->here), IO_THREADS, 0, c->stream>>>(k);
    c->launches++;
    CU(c, cudaGetLastError());
  }
  CU(c, cudaMemcpyAsync(c->host_small + 24, u, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
  return LSB_OK;
}

int unique_device(lsb_ctx* c, const char* fn, const lsb_key_column* cols, int32_t K, uint32_t unique_flags,
                  int64_t* index_out, int64_t* inverse_out, int64_t* counts_out, int64_t count, int64_t* num_unique,
                  void* stream, lsb_stats* st) {
  if (!c) return LSB_ERR_ARG;
  const std::string f(fn);
  std::vector<int> widths;
  int rc = check_columns(c, fn, cols, K, count, widths);
  if (rc) return rc;
  if (unique_flags & ~LSB_UNIQUE_CONSECUTIVE)
    return fail(c, LSB_ERR_ARG, f + ": unknown unique_flags " + std::to_string(unique_flags));
  if (!num_unique) return fail(c, LSB_ERR_ARG, f + ": num_unique is NULL");
  if (count) {
    int64_t* outs[3] = {index_out, inverse_out, counts_out};
    const char* names[3] = {"index_out", "inverse_out", "counts_out"};
    const size_t bytes = (size_t)count * sizeof(int64_t);
    for (int i = 0; i < 3; i++) {
      if ((rc = check_device_array(c, fn, outs[i], names[i], count))) return rc;
      if (!outs[i]) continue;
      for (int j = 0; j < i; j++)
        if (outs[j] && ranges_overlap(outs[i], bytes, outs[j], bytes))
          return fail(c, LSB_ERR_ARG, f + ": " + names[i] + " overlaps " + names[j]);
      for (int k = 0; k < K; k++)
        if (ranges_overlap(outs[i], bytes, cols[k].keys, (size_t)count * (widths[k] / 8)))
          return fail(c, LSB_ERR_ARG, f + ": " + names[i] + " overlaps column " + std::to_string(k));
    }
  }
  const std::vector<LexsortRound> rounds = column_rounds(c, widths);
  const bool sorted = !(unique_flags & LSB_UNIQUE_CONSECUTIVE);
  CU(c, cudaEventRecord(c->ev_caller, (cudaStream_t)stream));
  CU(c, cudaStreamWaitEvent(c->stream, c->ev_caller, 0));
  if ((rc = begin_call(c))) return rc;
  int passes = 0, subpasses = 0;
  if (sorted && (rc = sort_columns(c, cols, rounds, &passes, &subpasses))) return rc;
  if (count && (rc = launch_unique(c, cols, rounds, sorted, index_out, inverse_out, counts_out))) return rc;
  if ((rc = end_call(c, st, passes, subpasses))) return rc;
  *num_unique = count ? (int64_t)c->host_small[24] : 0;
  return LSB_OK;
}

}  // namespace

// =====================================================================================
// C ABI
// =====================================================================================
extern "C" {

int lsb_abi_version(void) { return LSB_ABI_VERSION; }

const char* lsb_status_string(int s) {
  switch (s) {
    case LSB_OK: return "ok";
    case LSB_ERR_ARG: return "bad argument";
    case LSB_ERR_CUDA: return "CUDA error";
    case LSB_ERR_NCCL: return "NCCL error";
    case LSB_ERR_STATE: return "wrong state";
    case LSB_ERR_NOMEM: return "out of memory";
    case LSB_ERR_VERIFY: return "verification failed";
  }
  return "unknown";
}

const char* lsb_last_error(const lsb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int lsb_tune(const char* key, int value) {
  if (!key) return LSB_ERR_ARG;
  const std::string k(key);
  if (k == "op_t1" && value >= 1 && value <= OP_MAX_T1) g_tune.op_t1 = value;
  else if (k == "op_cfg" && value >= 0 && value <= 1) g_tune.op_cfg = value;
  else if (k == "op_persist" && value >= 0) g_tune.op_persist = value;
  else if (k == "op_nx" && value >= 2 && value <= 8) g_tune.op_nx = value;
  else if (k == "op_lead" && value >= 1 && value <= 4) g_tune.op_lead = value;
  else if (k == "op_hints" && value >= 0 && value <= 15) g_tune.op_hints = value;
  else if (k == "op_ctas_mgpu" && value >= 0 && value <= 4) g_tune.op_ctas_mgpu = value;
  else if (k == "vparts" && value >= 1 && value <= LSB_MAX_PARTS) g_tune.vparts = value;
  else if (k == "vramp" && value >= 100 && value <= 300) g_tune.vramp = value;
  else if (k == "ex_ctas" && value >= 1 && value <= 8) g_tune.ex_ctas = value;
  else if (k == "ex_threads" && (value == 0 || value == 256 || value == 512)) g_tune.ex_threads = value;
  else if (k == "ex_u" && (value == 4 || value == 8)) g_tune.ex_u = value;
  else if (k == "timeout_ms" && value >= 1) g_tune.timeout_ms = value;
  else if (k == "pt_direct" && value >= 0 && value <= 1) g_tune.pt_direct = value;
  else if (k == "pt_chunks" && value >= 0 && value <= 4) g_tune.pt_chunks = value;
  else if (k == "pt_variant" && value >= 0 && value <= 1) g_tune.pt_variant = value;
  else if (k == "pt_pf_tiles" && value >= 0 && value <= 65536) g_tune.pt_pf_tiles = value;
  else return fail(nullptr, LSB_ERR_ARG, "lsb_tune: unknown key or value out of range: " + k);
  return LSB_OK;
}

#ifdef LSB_OP_PROF
// tools/ only: read and clear the one-pass kernel's stage clocks
int lsb_debug_prof(lsb_ctx* c, unsigned long long* out) {
  if (!c || !out) return LSB_ERR_ARG;
  CU(c, cudaMemcpy(out, c->op_prof, sizeof(unsigned long long) * OP_NPROF, cudaMemcpyDeviceToHost));
  CU(c, cudaMemset(c->op_prof, 0, sizeof(unsigned long long) * OP_NPROF));
  return LSB_OK;
}
#endif

int lsb_create(lsb_ctx** out, const lsb_config* cfg) {
  if (!out || !cfg) return fail(nullptr, LSB_ERR_ARG, "null argument");
  *out = nullptr;
  if (cfg->n < 0 || cfg->world_size < 1 || cfg->world_size > LSB_MAX_GPUS || cfg->world_rank < 0 ||
      cfg->world_rank >= cfg->world_size || cfg->radix_bits < 1 || cfg->radix_bits > 16 || cfg->ranks < 0)
    return fail(nullptr, LSB_ERR_ARG, "bad lsb_config (n >= 0, 1 <= world_size <= 8, 1 <= radix_bits <= 16)");
  if ((cfg->flags & LSB_FLAG_KEY_I64) && (cfg->flags & LSB_FLAG_KEY_F64))
    return fail(nullptr, LSB_ERR_ARG, "bad lsb_config: LSB_FLAG_KEY_I64 and LSB_FLAG_KEY_F64 exclude each other");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, LSB_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, LSB_ERR_ARG, "device ordinal out of range");

  lsb_ctx* c = new lsb_ctx();
  c->cfg = *cfg;
  c->tune = g_tune;
  if (c->tune.op_nx <= c->tune.op_lead) c->tune.op_nx = c->tune.op_lead + 1;
  if (c->cfg.ranks == 0) c->cfg.ranks = cfg->world_size;
  if (c->cfg.and_draws < 1) c->cfg.and_draws = 1;
  c->G = cfg->world_size;
  c->my = cfg->world_rank;
  c->n = cfg->n;
  // DistributedArray::create, mpi/mpi_lsbsort.cpp:144-149
  c->per = std::max<int64_t>(div_ceil(c->n, c->G), 1);
  c->here = c->per;
  if (c->per * c->my + c->here > c->n) c->here = c->n - c->per * c->my;
  if (c->here < 0) c->here = 0;
  c->first = c->per * c->my;
  c->per_stream = std::max<int64_t>(div_ceil(c->n, c->cfg.ranks), 1);
  c->npasses = num_passes(c, context_plan(c));

#define CUC(expr)                                                                        \
  do {                                                                                   \
    cudaError_t e_ = (expr);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      int code_ = (e_ == cudaErrorMemoryAllocation) ? LSB_ERR_NOMEM : LSB_ERR_CUDA;      \
      fail(nullptr, code_, std::string(#expr) + ": " + cudaGetErrorString(e_));          \
      lsb_destroy(c);                                                                    \
      return code_;                                                                      \
    }                                                                                    \
  } while (0)

  CUC(cudaSetDevice(cfg->device));
  CUC(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, cfg->device));
  CUC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CUC(cudaEventCreate(&c->ev_start));
  CUC(cudaEventCreate(&c->ev_stop));
  CUC(cudaEventCreateWithFlags(&c->ev_caller, cudaEventDisableTiming));
  const size_t shard_bytes = (size_t)std::max<int64_t>(c->per, 1) * sizeof(Elt);
  CUC(cudaMalloc(&c->buf[0], shard_bytes));
  CUC(cudaMalloc(&c->buf[1], shard_bytes));
  c->peer[0][c->my] = c->buf[0];
  c->peer[1][c->my] = c->buf[1];
  c->lookback_tiles = (size_t)div_ceil(c->per, c->tile) + 256 + 1;
  CUC(cudaMalloc(&c->lookback, c->lookback_tiles * 256 * sizeof(uint64_t)));
  CUC(cudaMemsetAsync(c->lookback, 0, c->lookback_tiles * 256 * sizeof(uint64_t), c->stream));
  CUC(cudaMalloc(&c->tile_counters, TILE_COUNTERS * sizeof(uint32_t)));
  CUC(cudaMalloc(&c->hist, sizeof(unsigned long long) * 256 * HIST_MAX_SUB));
  CUC(cudaMalloc(&c->scan_out, sizeof(int64_t) * 257 * HIST_MAX_SUB));
  CUC(cudaHostAlloc(&c->host_hist, sizeof(unsigned long long) * 256 * HIST_MAX_SUB, cudaHostAllocDefault));
  CUC(cudaMalloc(&c->hist16, sizeof(unsigned long long) * 65536 * 4));
  CUC(cudaMalloc(&c->starts16, sizeof(int64_t) * 65536 * 4));
  CUC(cudaMalloc(&c->dig_meta, sizeof(int) * 128));
  CUC(cudaMalloc(&c->skip_flags, sizeof(int) * 64));
  CUC(cudaHostAlloc(&c->host_skip, sizeof(int) * 64, cudaHostAllocDefault));
  CUC(cudaMalloc(&c->counts_all, sizeof(unsigned long long) * 65536 * c->G));
  CUC(cudaMalloc(&c->mybase, sizeof(int64_t) * 65536));
  // one-pass kernel: supertile scratch, piece table, control block, frontier table
#define LSB_PT_ATTR(V, O)                                                                                                     \
  CUC(cudaFuncSetAttribute(partition_kernel<TileCfg, V, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, TileCfg::SMEM));     \
  CUC(cudaFuncSetAttribute(partition_kernel<TileCfg, V, O>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  LSB_PT_ATTR(false, false)
  LSB_PT_ATTR(true, false)
  LSB_PT_ATTR(false, true)
  LSB_PT_ATTR(true, true)
#undef LSB_PT_ATTR
#define LSB_OP_ATTR(CFG, B, O)                                                                                       \
  CUC(cudaFuncSetAttribute(onepass_kernel<CFG, B, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, CFG::SMEM));     \
  CUC(cudaFuncSetAttribute(onepass_kernel<CFG, B, O>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  LSB_OP_ATTR(TileCfg, true, false)
  LSB_OP_ATTR(TileCfg, false, false)
  LSB_OP_ATTR(TileCfgS, true, false)
  LSB_OP_ATTR(TileCfgS, false, false)
  LSB_OP_ATTR(TileCfg, false, true)
  LSB_OP_ATTR(TileCfgS, false, true)
#undef LSB_OP_ATTR
  CUC(cudaFuncSetAttribute(digit_hist_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DH_SMEM));
  CUC(cudaFuncSetAttribute(digit_hist_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DH_SMEM));
  CUC(cudaFuncSetAttribute(digit_hist_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DH_SMEM));
  CUC(cudaFuncSetAttribute(digit_hist_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DH_SMEM));
  // every claimed one-pass item must belong to a resident CTA: residency of the instantiation this context launches
  if (c->tune.op_cfg == 1) {
    c->op_tile = TileCfgS::TILE;
    CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->op_resident, context_plan(c).korder ? onepass_kernel<TileCfgS, false, true> : onepass_kernel<TileCfgS, true, false>, TileCfgS::THREADS, TileCfgS::SMEM));
  } else {
    CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->op_resident, context_plan(c).korder ? onepass_kernel<TileCfg, false, true> : onepass_kernel<TileCfg, true, false>, TileCfg::THREADS, TileCfg::SMEM));
  }
  if (c->tune.op_persist > 0) {
    int max_persist = 0;
    CUC(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, cfg->device));
    CUC(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min<size_t>((size_t)c->tune.op_persist << 20, (size_t)max_persist)));
  }
  if (c->op_resident < 1) {
    fail(nullptr, LSB_ERR_CUDA, "one-pass kernel does not fit an SM");
    lsb_destroy(c);
    return LSB_ERR_CUDA;
  }
  {
    const int64_t tiles = div_ceil(c->per, c->op_tile);
    if (c->tune.op_t1 > tiles) c->tune.op_t1 = (int)std::max<int64_t>(1, tiles);
    c->op_S = (int64_t)c->tune.op_t1 * c->op_tile;
    const int64_t nsuper = div_ceil(c->per, c->op_S);
    const size_t words = 8 + (size_t)nsuper * (5 + 4 * 256);
    c->op_ctl_bytes = words * 4 + (size_t)c->tune.op_nx * (c->tune.op_t1 + 256) * 256 * sizeof(uint64_t);
    CUC(cudaMalloc(&c->op_ctl, c->op_ctl_bytes));
    CUC(cudaMalloc(&c->op_X, (size_t)c->tune.op_nx * c->op_S * sizeof(Elt)));
    CUC(cudaMalloc(&c->op_oc, (size_t)c->tune.op_nx * 256 * c->tune.op_t1 * sizeof(unsigned)));
    CUC(cudaMalloc(&c->op_F, sizeof(uint64_t) * 65536));
    CUC(cudaMalloc(&c->op_err, sizeof(unsigned)));
    CUC(cudaMalloc(&c->op_prof, sizeof(unsigned long long) * OP_NPROF));
    CUC(cudaMemsetAsync(c->op_prof, 0, sizeof(unsigned long long) * OP_NPROF, c->stream));
  }
  c->two_level = c->G > 1 || (cfg->flags & LSB_FLAG_TWO_LEVEL);
  c->V = c->two_level ? c->tune.vparts : 1;
  {
    // cut [0, per) into V parts: equal for small shards, a geometric ramp up and down otherwise (see Tuning::vramp)
    const int V = c->V;
    double w[LSB_MAX_PARTS], sum = 0;
    const bool ramp = c->per >= (int64_t)V * 4096 && c->tune.vramp > 100;
    for (int q = 0; q < V; q++) {
      w[q] = ramp ? std::pow(c->tune.vramp / 100.0, std::min(q, V - 1 - q)) : 1.0;
      sum += w[q];
    }
    const int64_t uniform = std::max<int64_t>(div_ceil(c->per, V), 1);
    double acc = 0;
    c->pstart[0] = 0;
    for (int q = 0; q < V; q++) {
      acc += w[q];
      int64_t e = ramp ? (int64_t)((double)c->per * (acc / sum)) / 32 * 32 : (int64_t)(q + 1) * uniform;
      if (q == V - 1 || e > c->per) e = c->per;
      c->pstart[q + 1] = std::max<int64_t>(e, c->pstart[q]);
      c->vpart_max = std::max<int64_t>(c->vpart_max, c->pstart[q + 1] - c->pstart[q]);
    }
    for (int q = V + 1; q <= LSB_MAX_PARTS; q++) c->pstart[q] = c->per;
    c->vpart_max = std::max<int64_t>(c->vpart_max, 1);
  }
  {
    int64_t segs[2 * (1 + LSB_MAX_PARTS)];
    uint32_t tls[2 * (1 + LSB_MAX_PARTS)];
    for (int i = 0; i <= c->V; i++) {
      const int64_t m = i == 0 ? c->here : part_len(c, i - 1);
      segs[2 * i] = 0;
      segs[2 * i + 1] = m;
      tls[2 * i] = 0;
      tls[2 * i + 1] = (uint32_t)div_ceil(m, c->tile);
    }
    CUC(cudaMalloc(&c->seg_start, sizeof(segs)));
    CUC(cudaMalloc(&c->seg_tiles, sizeof(tls)));
    CUC(cudaMemcpyAsync(c->seg_start, segs, sizeof(segs), cudaMemcpyHostToDevice, c->stream));
    CUC(cudaMemcpyAsync(c->seg_tiles, tls, sizeof(tls), cudaMemcpyHostToDevice, c->stream));
    CUC(cudaStreamSynchronize(c->stream));
  }
  {  // tables of the two-step shape (G == 1: one part = the shard) and of the virtual ranks
    const int V = c->V;
    CUC(cudaMalloc(&c->localbase_v, sizeof(int64_t) * 65536 * V));
    CUC(cudaMalloc(&c->bases_v, sizeof(int64_t) * 257 * 2 * V));
  }
  if (c->two_level) {
    const int V = c->V;
    CUC(cudaMalloc(&c->scratch[0], (size_t)(c->vpart_max + 64) * sizeof(Elt)));
    CUC(cudaMalloc(&c->scratch[1], (size_t)(c->vpart_max + 64) * sizeof(Elt)));
    CUC(cudaMalloc(&c->dense_local, sizeof(unsigned) * 65536 * V));
    CUC(cudaMalloc(&c->dense_mine, sizeof(unsigned) * 65536 * V));
    CUC(cudaMalloc(&c->next_dense, sizeof(unsigned) * 65536 * V * c->G));
    CUC(cudaMalloc(&c->c_all, sizeof(unsigned) * 65536 * V * c->G));
    CUC(cudaMalloc(&c->totals, sizeof(unsigned long long) * 65536));
    CUC(cudaMalloc(&c->fuse_live, sizeof(unsigned) * 64));
    CUC(cudaMalloc(&c->digit_base, sizeof(int64_t) * 65536));
    CUC(cudaMalloc(&c->mybase_v, sizeof(int64_t) * 65536 * V));
    int lo_prio = 0, hi_prio = 0;
    CUC(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
    CUC(cudaStreamCreateWithPriority(&c->xstream, cudaStreamNonBlocking, hi_prio));
    for (int q = 0; q < V; q++) {
      CUC(cudaEventCreateWithFlags(&c->ev_sorted[q], cudaEventDisableTiming));
      CUC(cudaEventCreateWithFlags(&c->ev_x[q], cudaEventDisableTiming));
    }
  }
  CUC(cudaMalloc(&c->small, sizeof(unsigned long long) * 64));
  CUC(cudaMalloc(&c->small_all, sizeof(unsigned long long) * 16 * LSB_MAX_GPUS));
  CUC(cudaMemsetAsync(c->small, 0, sizeof(unsigned long long) * 64, c->stream));
  CUC(cudaHostAlloc(&c->host_small, sizeof(unsigned long long) * (16 * LSB_MAX_GPUS + 64), cudaHostAllocDefault));
  CUC(cudaStreamSynchronize(c->stream));
#undef CUC
  *out = c;
  return LSB_OK;
}

void lsb_destroy(lsb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->cfg.device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->xstream) cudaStreamSynchronize(c->xstream);
  for (int b = 0; b < 2; b++)
    for (int g = 0; g < LSB_MAX_GPUS; g++)
      if (c->peer_open[b][g]) cudaIpcCloseMemHandle(c->peer[b][g]);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  for (auto ev : c->phase_ev) cudaEventDestroy(ev);
  for (auto ev : c->xev) cudaEventDestroy(ev);
  if (c->host_hist) cudaFreeHost(c->host_hist);
  void* dev[] = {c->seg_start, c->seg_tiles, c->hist, c->scan_out, c->buf[0], c->buf[1], c->lookback, c->tile_counters, c->hist16, c->starts16, c->dig_meta, c->skip_flags,
                 c->counts_all, c->mybase, c->op_ctl, c->op_X, c->op_oc, c->op_F, c->op_err, c->op_prof,
                 c->scratch[0], c->scratch[1], c->dense_local, c->dense_mine, c->next_dense, c->c_all, c->totals, c->fuse_live, c->digit_base,
                 c->mybase_v, c->localbase_v, c->bases_v, c->small, c->small_all};
  for (void* p : dev) cudaFree(p);
  for (int q = 0; q < LSB_MAX_PARTS; q++) {
    if (c->ev_sorted[q]) cudaEventDestroy(c->ev_sorted[q]);
    if (c->ev_x[q]) cudaEventDestroy(c->ev_x[q]);
  }
  if (c->xstream) cudaStreamDestroy(c->xstream);
  if (c->host_small) cudaFreeHost(c->host_small);
  if (c->host_skip) cudaFreeHost(c->host_skip);
  if (c->ev_start) cudaEventDestroy(c->ev_start);
  if (c->ev_stop) cudaEventDestroy(c->ev_stop);
  if (c->ev_caller) cudaEventDestroy(c->ev_caller);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int lsb_comm_unique_id(void* id_out) {
  if (!id_out) return LSB_ERR_ARG;
  static_assert(sizeof(ncclUniqueId) == LSB_COMM_ID_BYTES, "ncclUniqueId size");
  if (!g_nccl.load()) return fail(nullptr, LSB_ERR_NCCL, g_nccl.error);
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) return fail(nullptr, LSB_ERR_NCCL, std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r));
  memcpy(id_out, &id, sizeof(id));
  return LSB_OK;
}

int lsb_comm_init(lsb_ctx* c, const void* id_bytes) {
  if (!c || !id_bytes) return LSB_ERR_ARG;
  if (c->G == 1) { c->comm_ready = true; return LSB_OK; }
  if (c->comm_ready) return fail(c, LSB_ERR_STATE, "communicator already initialised");
  if (!g_nccl.load()) return fail(c, LSB_ERR_NCCL, g_nccl.error);
  CU(c, cudaSetDevice(c->cfg.device));
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof(id));
  NC(c, g_nccl.CommInitRank(&c->comm, c->G, id, c->my));
  // exchange CUDA IPC handles of both shards through the communicator itself
  struct Handles { cudaIpcMemHandle_t h[2]; };
  static_assert(sizeof(Handles) == 128, "ipc handle size");
  Handles mine;
  CU(c, cudaIpcGetMemHandle(&mine.h[0], c->buf[0]));
  CU(c, cudaIpcGetMemHandle(&mine.h[1], c->buf[1]));
  unsigned char* d_h = nullptr;
  CU(c, cudaMalloc(&d_h, sizeof(Handles) * (c->G + 1)));
  CU(c, cudaMemcpyAsync(d_h, &mine, sizeof(mine), cudaMemcpyHostToDevice, c->stream));
  NC(c, g_nccl.AllGather(d_h, d_h + sizeof(Handles), sizeof(Handles), ncclUint8, c->comm, c->stream));
  std::vector<Handles> all(c->G);
  CU(c, cudaMemcpyAsync(all.data(), d_h + sizeof(Handles), sizeof(Handles) * c->G, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  CU(c, cudaFree(d_h));
  for (int g = 0; g < c->G; g++) {
    if (g == c->my) continue;
    for (int b = 0; b < 2; b++) {
      void* p = nullptr;
      CU(c, cudaIpcOpenMemHandle(&p, all[g].h[b], cudaIpcMemLazyEnablePeerAccess));
      c->peer[b][g] = reinterpret_cast<Elt*>(p);
      c->peer_open[b][g] = true;
    }
  }
  c->comm_ready = true;
  return LSB_OK;
}

int lsb_barrier(lsb_ctx* c) {
  int rc = check_ready(c);
  if (rc) return rc;
  CU(c, cudaSetDevice(c->cfg.device));
  if ((rc = stream_barrier(c))) return rc;
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int lsb_shard_info(const lsb_ctx* c, int64_t* per, int64_t* here, int64_t* first_global) {
  if (!c) return LSB_ERR_ARG;
  if (per) *per = c->per;
  if (here) *here = c->here;
  if (first_global) *first_global = c->first;
  return LSB_OK;
}

int lsb_num_passes(const lsb_ctx* c) { return c ? c->npasses : LSB_ERR_ARG; }

int lsb_digit_bits(const lsb_ctx* c, int digit) {
  if (!c || digit < 0 || digit >= c->npasses) return LSB_ERR_ARG;
  return plan_pass(c, context_plan(c), digit).bits;
}

int lsb_generate(lsb_ctx* c) {
  if (!c) return LSB_ERR_ARG;
  CU(c, cudaSetDevice(c->cfg.device));
  c->cur = 0;
  if (c->here > 0) {
    GenArgs a;
    a.dst = c->buf[0];
    a.first_global = c->first;
    a.count = c->here;
    a.per_stream = c->per_stream;
    a.seed_base = c->cfg.seed_base;
    a.key_mask = c->cfg.key_mask;
    a.and_draws = c->cfg.and_draws;
    u128 m, p;
    pcg_jump_coeffs((u128)32 * (u128)c->cfg.and_draws, m, p);
    a.row_mult_hi = (uint64_t)(m >> 64);
    a.row_mult_lo = (uint64_t)m;
    a.row_plus_hi = (uint64_t)(p >> 64);
    a.row_plus_lo = (uint64_t)p;
    const int64_t warps = div_ceil(c->here, 32 * GEN_ROWS);
    const int64_t blocks = div_ceil(warps * 32, GEN_THREADS);
    generate_kernel<<<(unsigned)blocks, GEN_THREADS, 0, c->stream>>>(a);
    CU(c, cudaGetLastError());
  }
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int lsb_upload(lsb_ctx* c, const lsb_elt* host, int64_t off, int64_t count) {
  if (!c || (!host && count) || off < 0 || count < 0 || off + count > c->per) return fail(c, LSB_ERR_ARG, "lsb_upload: range");
  CU(c, cudaSetDevice(c->cfg.device));
  if (count) CU(c, cudaMemcpyAsync(c->buf[c->cur] + off, host, (size_t)count * sizeof(Elt), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int lsb_download(lsb_ctx* c, lsb_elt* host, int64_t off, int64_t count) {
  if (!c || (!host && count) || off < 0 || count < 0 || off + count > c->per) return fail(c, LSB_ERR_ARG, "lsb_download: range");
  CU(c, cudaSetDevice(c->cfg.device));
  if (count) CU(c, cudaMemcpyAsync(host, c->buf[c->cur] + off, (size_t)count * sizeof(Elt), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int lsb_device_ptr(lsb_ctx* c, void** ptr) {
  if (!c || !ptr) return LSB_ERR_ARG;
  *ptr = c->buf[c->cur];
  return LSB_OK;
}

int lsb_host_alloc(void** ptr, int64_t bytes) {
  if (!ptr || bytes < 0) return LSB_ERR_ARG;
  cudaError_t e = cudaHostAlloc(ptr, (size_t)std::max<int64_t>(bytes, 1), cudaHostAllocDefault);
  if (e != cudaSuccess) return fail(nullptr, LSB_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
  return LSB_OK;
}

int lsb_host_free(void* ptr) {
  if (!ptr) return LSB_OK;
  return cudaFreeHost(ptr) == cudaSuccess ? LSB_OK : LSB_ERR_CUDA;
}

int lsb_sort(lsb_ctx* c, lsb_stats* st) {
  const int rc = check_ready(c);
  return rc ? rc : sort_shard(c, context_plan(c), st);
}

int lsb_pass(lsb_ctx* c, int digit, lsb_stats* st) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (digit < 0 || digit >= c->npasses) return fail(c, LSB_ERR_ARG, "lsb_pass: digit out of range");
  CU(c, cudaSetDevice(c->cfg.device));
  if ((rc = begin_call(c))) return rc;
  c->dense_ready_digit = -1;
  int subpasses = 0;
  if (!c->two_level) rc = passes_single(c, context_plan(c), digit, digit + 1, &subpasses);
  else rc = pass_global(c, context_plan(c), digit, &subpasses, false);
  if (rc) return rc;
  return end_call(c, st, 1, subpasses);
}

int lsb_sort_host(lsb_ctx* c, const lsb_elt* host_in, lsb_elt* host_out, int64_t count, lsb_stats* st) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (count != c->here || (count && (!host_in || !host_out))) return fail(c, LSB_ERR_ARG, "lsb_sort_host: count must equal this shard's size");
  CU(c, cudaSetDevice(c->cfg.device));
  c->cur = 0;
  if (count) CU(c, cudaMemcpyAsync(c->buf[0], host_in, (size_t)count * sizeof(Elt), cudaMemcpyHostToDevice, c->stream));
  if ((rc = lsb_sort(c, st))) return rc;
  if (count) CU(c, cudaMemcpyAsync(host_out, c->buf[c->cur], (size_t)count * sizeof(Elt), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

int lsb_sort_device(lsb_ctx* c, const uint64_t* keys_in, const uint64_t* vals_in, uint64_t* keys_out, uint64_t* vals_out,
                    int64_t count, void* stream, lsb_stats* st) {
  return sort_device(c, "lsb_sort_device", LSB_KEY_CONTEXT, keys_in, vals_in, keys_out, vals_out, count, stream, st);
}

int lsb_sort_device_typed(lsb_ctx* c, uint32_t key_type, const void* keys_in, const uint64_t* vals_in, void* keys_out,
                          uint64_t* vals_out, int64_t count, void* stream, lsb_stats* st) {
  return sort_device(c, "lsb_sort_device_typed", key_type, keys_in, vals_in, keys_out, vals_out, count, stream, st);
}

int lsb_sort_segments_device(lsb_ctx* c, const uint64_t* keys_in, const uint64_t* vals_in, uint64_t* keys_out,
                             uint64_t* vals_out, int64_t count, const int64_t* seg_offsets, int64_t num_segments,
                             uint32_t seg_flags, void* stream, lsb_stats* st) {
  return sort_segments_device(c, "lsb_sort_segments_device", LSB_KEY_CONTEXT, keys_in, vals_in, keys_out, vals_out, count,
                              seg_offsets, num_segments, seg_flags, stream, st);
}

int lsb_sort_segments_device_typed(lsb_ctx* c, uint32_t key_type, const void* keys_in, const uint64_t* vals_in,
                                   void* keys_out, uint64_t* vals_out, int64_t count, const int64_t* seg_offsets,
                                   int64_t num_segments, uint32_t seg_flags, void* stream, lsb_stats* st) {
  return sort_segments_device(c, "lsb_sort_segments_device_typed", key_type, keys_in, vals_in, keys_out, vals_out, count,
                              seg_offsets, num_segments, seg_flags, stream, st);
}

int lsb_lexsort_device(lsb_ctx* c, const lsb_key_column* columns, int32_t num_columns, const uint64_t* vals_in,
                       uint64_t* vals_out, int64_t count, void* stream, lsb_stats* st) {
  return lexsort_device(c, "lsb_lexsort_device", columns, num_columns, vals_in, vals_out, count, stream, st);
}

int lsb_unique_device(lsb_ctx* c, const lsb_key_column* columns, int32_t num_columns, uint32_t unique_flags,
                      int64_t* index_out, int64_t* inverse_out, int64_t* counts_out, int64_t count, int64_t* num_unique,
                      void* stream, lsb_stats* st) {
  return unique_device(c, "lsb_unique_device", columns, num_columns, unique_flags, index_out, inverse_out, counts_out,
                       count, num_unique, stream, st);
}

// The two test hooks run the PRODUCTION count and scan kernels of the pass shape in use.
int lsb_histogram(lsb_ctx* c, int digit, int64_t* host_counts) {
  if (!c || !host_counts || digit < 0 || digit >= c->npasses) return fail(c, LSB_ERR_ARG, "lsb_histogram: argument");
  CU(c, cudaSetDevice(c->cfg.device));
  const KeyPlan k = context_plan(c);
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits, zero = 0;
  CU(c, cudaMemsetAsync(c->hist16, 0, sizeof(unsigned long long) * nb, c->stream));
  int rc = launch_digit_hist(c, k.korder, c->buf[c->cur], c->here, &p.shift, &p.bits, &zero, 1, c->hist16, false);
  if (rc) return rc;
  CU(c, cudaMemcpyAsync(host_counts, c->hist16, sizeof(int64_t) * nb, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  if (!c->two_level && !(c->cfg.flags & LSB_FLAG_ONE_PASS) && c->here > 0) {
    // the default shape counts 8-bit sub-digits (subdigit_hist_kernel): its histograms must be the marginals of
    // the digit's counts just returned, so a caller that checks those against the reference checks both kernels
    SubPass subs[2];
    int ns = 0;
    if (p.lo_bits) subs[ns++] = {p.shift, p.lo_bits};
    subs[ns++] = {p.shift + p.lo_bits, p.hi_bits};
    if ((rc = launch_subdigit_hist(c, k.korder, c->buf[c->cur], subs, ns))) return rc;
    CU(c, cudaMemcpyAsync(c->host_hist, c->hist, sizeof(unsigned long long) * 256 * ns, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    std::vector<unsigned long long> lo(256, 0), hi(256, 0);
    for (int d = 0; d < nb; d++) {
      lo[d & ((1 << p.lo_bits) - 1)] += (unsigned long long)host_counts[d];
      hi[d >> p.lo_bits] += (unsigned long long)host_counts[d];
    }
    for (int b = 0; b < 256; b++) {
      const bool lo_ok = !p.lo_bits || c->host_hist[b] == lo[b];
      const bool hi_ok = c->host_hist[(ns - 1) * 256 + b] == hi[b];
      if (!lo_ok || !hi_ok) return fail(c, LSB_ERR_STATE, "lsb_histogram: sub-digit histograms are not the marginals of the digit counts");
    }
  }
  return LSB_OK;
}

int lsb_starts(lsb_ctx* c, int digit, int64_t* host_starts) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (!host_starts || digit < 0 || digit >= c->npasses) return fail(c, LSB_ERR_ARG, "lsb_starts: argument");
  CU(c, cudaSetDevice(c->cfg.device));
  const KeyPlan k = context_plan(c);
  const PassPlan p = plan_pass(c, k, digit);
  const int nb = 1 << p.bits, zero = 0;
  const int64_t* src;
  if (c->two_level) {
    // a shard's first element of digit d is its first part's first element of digit d
    if ((rc = count_parts(c, k, digit))) return rc;
    if ((rc = part_offsets(c, k, digit))) return rc;
    src = c->mybase_v;
  } else {
    CU(c, cudaMemsetAsync(c->hist16, 0, sizeof(unsigned long long) * nb, c->stream));
    if ((rc = launch_digit_hist(c, k.korder, c->buf[c->cur], c->here, &p.shift, &p.bits, &zero, 1, c->hist16, false))) return rc;
    if ((rc = launch_scan(c, c->hist16, nb, 1, 0, c->mybase, nullptr))) return rc;
    src = c->mybase;
  }
  CU(c, cudaMemcpyAsync(host_starts, src, sizeof(int64_t) * nb, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return LSB_OK;
}

static int local_verify(lsb_ctx* c) {
  // small[40..44] = checksum[4], violations
  CU(c, cudaMemsetAsync(c->small + 40, 0, 8 * sizeof(unsigned long long), c->stream));
  if (c->here > 0) {
    int grid = (int)std::min<int64_t>((int64_t)c->num_sms * 8, div_ceil(c->here, 256));
    const uint32_t korder = context_plan(c).korder;
    if (korder) verify_kernel<true><<<grid, 256, 0, c->stream>>>(c->buf[c->cur], c->here, c->small + 40, korder);
    else verify_kernel<false><<<grid, 256, 0, c->stream>>>(c->buf[c->cur], c->here, c->small + 40, 0);
    CU(c, cudaGetLastError());
  }
  return LSB_OK;
}

int lsb_checksum(lsb_ctx* c, uint64_t out[4]) {
  if (!c || !out) return LSB_ERR_ARG;
  CU(c, cudaSetDevice(c->cfg.device));
  int rc = local_verify(c);
  if (rc) return rc;
  CU(c, cudaMemcpyAsync(c->host_small, c->small + 40, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  for (int i = 0; i < 4; i++) out[i] = c->host_small[i];
  return LSB_OK;
}

int lsb_verify_device(lsb_ctx* c, lsb_verify* out) {
  int rc = check_ready(c);
  if (rc) return rc;
  if (!out) return LSB_ERR_ARG;
  CU(c, cudaSetDevice(c->cfg.device));
  if ((rc = local_verify(c))) return rc;
  // record = {checksum[4], violations, here, first.key, first.val, last.key, last.val}
  unsigned long long* rec = c->small + 48;  // 10 words used, 16 reserved
  CU(c, cudaMemcpyAsync(rec, c->small + 40, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
  const unsigned long long here = (unsigned long long)c->here;
  CU(c, cudaMemcpyAsync(rec + 5, &here, sizeof(here), cudaMemcpyHostToDevice, c->stream));
  if (c->here > 0) {
    CU(c, cudaMemcpyAsync(rec + 6, c->buf[c->cur], sizeof(Elt), cudaMemcpyDeviceToDevice, c->stream));
    CU(c, cudaMemcpyAsync(rec + 8, c->buf[c->cur] + (c->here - 1), sizeof(Elt), cudaMemcpyDeviceToDevice, c->stream));
  }
  const unsigned long long* all = rec;
  if (c->G > 1) {
    NC(c, g_nccl.AllGather(rec, c->small_all, 16, ncclUint64, c->comm, c->stream));
    all = c->small_all;
  }
  CU(c, cudaMemcpyAsync(c->host_small, all, sizeof(unsigned long long) * 16 * c->G, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  memset(out, 0, sizeof(*out));
  bool have_prev = false;
  uint64_t pk = 0, pv = 0;
  for (int g = 0; g < c->G; g++) {
    const unsigned long long* r = c->host_small + 16 * g;
    out->checksum[0] += r[0];
    out->checksum[1] ^= r[1];
    out->checksum[2] ^= r[2];
    out->checksum[3] += r[3];
    out->order_violations += (int64_t)r[4];
    out->elements += (int64_t)r[5];
    if (r[5] == 0) continue;
    const uint64_t fk = order_key(r[6], c->cfg.flags);
    if (have_prev && (pk > fk || (pk == fk && pv >= r[7]))) out->order_violations++;
    pk = order_key(r[8], c->cfg.flags);
    pv = r[9];
    have_prev = true;
  }
  if (out->order_violations) return fail(c, LSB_ERR_VERIFY, "shards are not strictly increasing in (key,val)");
  return LSB_OK;
}

}  // extern "C"
