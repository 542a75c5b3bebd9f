/*
 * lsbsort.h -- C ABI of the B200-native distributed LSD radix sort.
 *
 * This is the drop-in boundary for the one hot path of ronawho/distributed-lsb:
 *   mySort(A, B)              mpi/mpi_lsbsort.cpp:580-585
 *   globalShuffle(A, B, d)    mpi/mpi_lsbsort.cpp:481-577
 * plus the two things main() does around it that define the workload and the answer:
 *   the pcg64(rank) generator mpi/mpi_lsbsort.cpp:650-656
 *   the verifier              mpi/mpi_lsbsort.cpp:710-739
 * The reference has no plugin/FFI interface (everything is one translation unit), so
 * the seam is where main() calls mySort (mpi/mpi_lsbsort.cpp:691).  INTEGRATION.md shows
 * the few lines a maintainer adds to mpi_lsbsort.cpp to call through this header.
 *
 * Process model: one process (= one MPI rank of the reference) per GPU.  The
 * reference's DistributedArray<SortElement> (mpi/mpi_lsbsort.cpp:90-161) becomes a
 * device-resident pair of shards A/B owned by the context: shard g holds the global
 * indices [g*per, g*per+here), per = ceil(n/G), here clamped exactly as
 * DistributedArray::create does (:144-149).
 *
 * Element ABI: 16 bytes, { uint64 key; uint64 val; }, key first, little endian --
 * identical to SortElement (mpi/mpi_lsbsort.cpp:29-32).
 *
 * Errors: every call returns LSB_OK (0) or a negative lsb_status; the text of the
 * CUDA/NCCL failure is kept in the context (lsb_last_error).  The reference aborts on
 * error instead ("errors returned by MPI calls do not need to be handled", :17-19).
 * There is NO CPU fallback: without a CUDA device lsb_create fails with LSB_ERR_CUDA.
 *
 * Threading: a context is not thread-safe, but contexts share no state: different contexts (also on one GPU)
 * may be used from different threads at the same time.  Calls are synchronous on return.
 */
#ifndef LSBSORT_H
#define LSBSORT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSB_ABI_VERSION 1
#define LSB_MAX_GPUS 8
#define LSB_MAX_SUBPASSES 32
#define LSB_MAX_PARTS 16   /* parts per shard of the multi-GPU pass (virtual ranks) */
#define LSB_COMM_ID_BYTES 128

typedef enum {
  LSB_OK = 0,
  LSB_ERR_ARG = -1,     /* bad argument / configuration                         */
  LSB_ERR_CUDA = -2,    /* CUDA runtime failure (text in lsb_last_error)        */
  LSB_ERR_NCCL = -3,    /* NCCL failure                                         */
  LSB_ERR_STATE = -4,   /* call made in the wrong state (e.g. comm not set up)  */
  LSB_ERR_NOMEM = -5,   /* device or host allocation failed                     */
  LSB_ERR_VERIFY = -6   /* lsb_verify_device found the shard(s) unsorted        */
} lsb_status;

/* one 16-byte record == SortElement, mpi/mpi_lsbsort.cpp:29-32 */
typedef struct lsb_elt {
  uint64_t key;
  uint64_t val;
} lsb_elt;

typedef struct lsb_ctx lsb_ctx;

/*
 * Knobs of the reference driver (mpi/mpi_lsbsort.cpp:594-611) plus what `mpirun -n R`
 * and `#define RADIX` (:21) fix at launch/compile time there.
 */
typedef struct lsb_config {
  int64_t n;            /* --n: total number of elements over all shards (:594-598)        */
  int32_t ranks;        /* R of `mpirun -n R`: number of pcg64 streams of the generator;
                           stream r = pcg64(seed_base + r) fills global slots
                           [r*ceil(n/R), (r+1)*ceil(n/R)) (:144-149,:650-656). 0 => world_size */
  int32_t world_size;   /* G: number of GPUs == number of processes                        */
  int32_t world_rank;   /* g: which shard this process owns                                */
  int32_t device;       /* CUDA device ordinal for this process                            */
  int32_t radix_bits;   /* RADIX (:21): 1..16; the reference uses 16 (4 passes)            */
  int32_t and_draws;    /* 1 = reference; k>1: key = AND of k successive draws (skew)      */
  uint64_t seed_base;   /* 0 = reference (pcg64(myRank), :650)                             */
  uint64_t key_mask;    /* ~0 = reference; 0xFFFFFF = "only low 24 bits random" skew       */
  uint32_t flags;       /* LSB_FLAG_*                                                      */
  uint32_t reserved;
} lsb_config;

#define LSB_FLAG_NONE 0u
#define LSB_FLAG_PHASE_EVENTS 1u /* record a CUDA event after every kernel of lsb_sort      */
#define LSB_FLAG_TWO_LEVEL 2u    /* run the multi-GPU pass shape (virtual ranks: per-part counts,
                                    digit-major / rank-minor scan, part sort + exchange kernel)
                                    even when world_size == 1                                  */
#define LSB_FLAG_ONE_PASS 4u     /* sort a 9..16-bit digit with the one-pass kernel: every element moves through
                                    HBM once per reference pass (L2-resident supertiles) instead of twice (two
                                    stable 8-bit counting-sort steps, the default); same permutation          */
#define LSB_FLAG_NO_SKIP 8u      /* do not skip passes whose digit is constant over the shard
                                    (a stable pass on a constant digit is the identity; the
                                    reference always runs it; chpl passes nBits for the same
                                    purpose, chpl/arkouda-radix-sort.chpl:70,78)              */
/*
 * Key orders.  Without a type flag the key is a uint64, sorted ascending.  The result of every
 * sort is "stable, ascending by order_key(key)", where
 *   uint64:            order_key(k) = k
 *   LSB_FLAG_KEY_I64:  order_key(k) = k ^ 2^63                 (two's-complement int64)
 *   LSB_FLAG_KEY_F64:  -0.0 is first read as +0.0; any NaN (exponent all ones, mantissa != 0,
 *                      either sign) maps to ~0; every other value k to k ^ (sign ? ~0 : 2^63)
 *   LSB_FLAG_DESCENDING (with either type flag or neither): ~order_key_ascending(k)
 * That is the order of np.argsort(x, kind="stable") and torch.sort(x, stable=True[, descending=True]):
 * NaNs last ascending and first descending, -0.0 == +0.0, equal keys in input order (for G > 1:
 * global index order, also descending).  The sort never rewrites key bits: the output holds the
 * input's records permuted (-0.0 stays -0.0, NaN payloads survive), so lsb_checksum is unchanged.
 * lsb_histogram, lsb_starts and lsb_pass count and move by the digits of order_key(key), a pass
 * whose digit of order_key is constant is skipped, and lsb_verify_device checks that
 * (order_key(key), val) strictly increases.  KEY_I64 | KEY_F64 together: LSB_ERR_ARG from lsb_create.
 * Definition: distributed-lsb_b200/csrc/lsb_keyorder.cuh.
 */
#define LSB_FLAG_KEY_I64 16u     /* key is a two's-complement int64                             */
#define LSB_FLAG_KEY_F64 32u     /* key is an IEEE-754 binary64                                 */
#define LSB_FLAG_DESCENDING 64u  /* largest first                                               */

/*
 * Key types of lsb_sort_device_typed / lsb_sort_segments_device_typed.  LSB_KEY_CONTEXT is the 8-byte key the
 * context's flags name.  The others are narrow keys of W = 32 or 16 bits, W / 8 bytes each in the caller's arrays,
 * aligned to their own width:
 *   LSB_KEY_U32 / LSB_KEY_U16:  order k
 *   LSB_KEY_I32 / LSB_KEY_I16:  order k ^ signbit (two's complement)
 *   LSB_KEY_F32 / LSB_KEY_F16 / LSB_KEY_BF16 (exponent/mantissa 8/23, 5/10, 8/7 bits): the LSB_FLAG_KEY_F64 rule at
 *     width W: -0 as +0, every NaN as all ones, any other value k ^ (sign ? all ones : signbit)
 *   LSB_FLAG_DESCENDING: the complement of that within W bits.
 * The order is numpy's and torch's stable one, as for the 8-byte keys.  A narrow key travels in the record's key word
 * as (uint64)k << 32 | order_W(k); the sort takes ceil(W / radix_bits) passes over the low W bits only (uint64
 * ascending: the order was applied by the pack), and the key written back is the word's high half, so key bits are
 * never rewritten.  A narrow type needs a context without LSB_FLAG_KEY_I64 / LSB_FLAG_KEY_F64.
 */
#define LSB_KEY_CONTEXT 0   /* 8-byte key ordered by the context's flags: exactly lsb_sort_device */
#define LSB_KEY_U32 1
#define LSB_KEY_I32 2
#define LSB_KEY_F32 3
#define LSB_KEY_U16 4
#define LSB_KEY_I16 5
#define LSB_KEY_F16 6
#define LSB_KEY_BF16 7

/* what lsb_sort / lsb_pass measured, device time from CUDA events on the sort stream */
typedef struct lsb_stats {
  double device_ms;       /* whole call: first kernel start -> last kernel end             */
  int32_t passes;         /* reference passes run (N_DIGITS, :22)                          */
  int32_t subpasses;      /* scatter-kernel launches (2 per 16-bit pass and part; 1 with ONE_PASS) */
  int32_t skipped;        /* steps (ONE_PASS: passes) skipped because their digit was constant */
  int32_t reserved0;
  int64_t elements;       /* elements of THIS shard that took part                         */
  double hist_ms;         /* count kernels (needs LSB_FLAG_PHASE_EVENTS, else 0)           */
  double scan_ms;         /* scans + collectives on counts                                 */
  double partition_ms;    /* partition (scatter) kernels                                   */
  double exchange_ms;     /* G > 1: exchange kernels (NVLink stores)                       */
  double subpass_ms[LSB_MAX_SUBPASSES]; /* per partition-kernel launch                     */
  int64_t sent[LSB_MAX_GPUS]; /* last pass: elements this shard sent to each GPU (:553-554) */
  int64_t partition_launches;
  int64_t partition_elements; /* elements moved by all partition launches of the call          */
  int64_t kernel_launches; /* all kernels launched by the call                             */
} lsb_stats;

typedef struct lsb_verify {
  int64_t order_violations;  /* i with (order_key(key),val)[i-1] >= (...)[i], within and across shards */
  int64_t elements;          /* global element count seen                                   */
  uint64_t checksum[4];      /* global multiset hash, see lsb_checksum                      */
} lsb_verify;

/* ---- lifetime ------------------------------------------------------------------ */

int lsb_abi_version(void);

/* DistributedArray<SortElement>::create for A and B (:138-161,:638-639): allocates both
 * device shards and every scratch table once.  The reference re-allocates its count and
 * send/recv buffers inside every pass (:489-490,:511-516,:538-543); here nothing is
 * allocated after lsb_create. */
int lsb_create(lsb_ctx** out, const lsb_config* cfg);
void lsb_destroy(lsb_ctx* ctx);
const char* lsb_last_error(const lsb_ctx* ctx);
const char* lsb_status_string(int status);

/* Experiment knob (profiling sweeps only; the defaults are what bench.py measures): sets a
 * process-wide tunable read by the NEXT lsb_create.  Keys: one-pass kernel -- "op_cfg" (tile
 * shape: 0 = 512 threads x 11 elements, 1 = 256 x 11), "op_t1" (tiles per supertile, 1..256),
 * "op_nx" (supertile scratch slots), "op_lead" (supertiles between a tile and its use),
 * "op_hints" (L2 eviction hints, bit mask), "op_persist" (MiB of persisting L2),
 * "op_ctas_mgpu" (one-pass CTAs per SM while an exchange kernel shares the GPU), "timeout_ms"
 * (watchdog); multi-GPU pass -- "vparts" (parts per shard), "vramp" (size ratio of neighbouring
 * parts x 100), "ex_ctas", "ex_threads", "ex_u" (exchange kernel shape); 8-bit scatter kernel --
 * "pt_direct" (1 = tile index from blockIdx and the tile load issued first, 0 = tiles handed out
 * by a ticket counter), "pt_chunks" (log2 of the bulk copies a tile arrives in, 0..4), "pt_variant" (1 = the CTA of tile t
 * also bulk-prefetches tile t + pt_pf_tiles into L2 [default], 0 = no prefetch), "pt_pf_tiles"
 * (prefetch distance in tiles, 0 = half the SM count).
 * Unknown key / bad value: LSB_ERR_ARG. */
int lsb_tune(const char* key, int value);

/* ---- multi-GPU wiring (MPI_Init / MPI_COMM_WORLD, :588,:613-616) ----------------- */

/* rank 0 calls lsb_comm_unique_id and hands the 128 bytes to every process (any
 * out-of-band channel); then every process calls lsb_comm_init.  It creates the NCCL
 * communicator used for the per-pass count all-gather (replaces the count transpose
 * MPI_Alltoallv + MPI_Exscan, :327-414) and maps every peer's A/B shards over
 * NVLink (CUDA IPC) so the scatter kernel can store straight into the destination
 * shard (replaces pack + MPI_Alltoallv + unpack, :530-576).  Not needed when G == 1. */
int lsb_comm_unique_id(void* id_out /* LSB_COMM_ID_BYTES */);
int lsb_comm_init(lsb_ctx* ctx, const void* id /* LSB_COMM_ID_BYTES */);

/* MPI_Barrier(MPI_COMM_WORLD) (:688,:693): every GPU has finished everything queued on
 * its sort stream.  Collective; a plain device synchronise when G == 1. */
int lsb_barrier(lsb_ctx* ctx);

/* ---- data ---------------------------------------------------------------------- */

/* per = numElementsPerRank (:103), here = numElementsHere (:104), first = r*per */
int lsb_shard_info(const lsb_ctx* ctx, int64_t* per, int64_t* here, int64_t* first_global);

/* the generator loop (:650-656) for this shard, on the device, bit-exact with pcg64 */
int lsb_generate(lsb_ctx* ctx);

/* caller-supplied data instead of lsb_generate: copy `count` elements from host memory
 * into this shard starting at local index local_off (A.localPart()[local_off..]) */
int lsb_upload(lsb_ctx* ctx, const lsb_elt* host, int64_t local_off, int64_t count);
/* copy elements of the current (sorted or not) shard back to host memory */
int lsb_download(lsb_ctx* ctx, lsb_elt* host, int64_t local_off, int64_t count);

/* device pointer of the shard that currently holds the data (after lsb_sort: the result) */
int lsb_device_ptr(lsb_ctx* ctx, void** ptr);

/* pinned host memory helpers for the host-buffer path */
int lsb_host_alloc(void** ptr, int64_t bytes);
int lsb_host_free(void* ptr);

/* ---- the hot path ---------------------------------------------------------------- */

/* mySort (:580-585): all ceil(64/radix_bits) passes, least significant digit first, on the digits
 * of order_key(key) (see the key orders above); on return the shard holds its slice of the
 * globally, stably sorted array.
 * Collective: every process must call it.  stats may be NULL. */
int lsb_sort(lsb_ctx* ctx, lsb_stats* stats);

/* globalShuffle(A, B, digit) (:481-577): one stable pass on digit `digit` of order_key(key).
 * Collective. */
int lsb_pass(lsb_ctx* ctx, int digit, lsb_stats* stats);

/* host-buffer form of mySort for one process: upload `count` elements (must equal
 * `here`), sort, download into host_out.  This is the end-to-end entry point a caller
 * with data in host memory uses; copies are inside the call. Collective. */
int lsb_sort_host(lsb_ctx* ctx, const lsb_elt* host_in, lsb_elt* host_out, int64_t count,
                  lsb_stats* stats);

/* mySort on device memory: pack keys_in[0..count) and vals_in (NULL: the global input index, i.e. the stable argsort)
 * into this shard, sort as lsb_sort does, and write the sorted keys and/or values to keys_out / vals_out (either may be
 * NULL, not both).  count must equal `here`; all pointers are device memory of this context's device, 8-byte aligned;
 * outputs may alias inputs (in place), keys_out and vals_out must not overlap.  The library's stream first waits for
 * everything already queued on `stream` (a cudaStream_t of the caller, NULL = the legacy default stream), so a producer
 * on that stream needs no synchronise.  Synchronous on return; afterwards the shard holds the sorted records, so
 * lsb_verify_device / lsb_checksum / lsb_download work as after lsb_sort.  stats describes the sort between pack and
 * unpack, as lsb_sort_host's excludes its copies.  With count == 0 the pointers are not looked at.  Bad pointers or
 * count: LSB_ERR_ARG.  Collective. */
int lsb_sort_device(lsb_ctx* ctx, const uint64_t* keys_in, const uint64_t* vals_in, uint64_t* keys_out,
                    uint64_t* vals_out, int64_t count, void* stream, lsb_stats* stats);

/* Segmented sort on device memory: segment s is the input positions [seg_offsets[s], seg_offsets[s+1]) (num_segments
 * segments, empty ones allowed), and the result is the stable sort by (s, order_key(key)): every segment sorted in the
 * context's key order, the segments themselves in ascending order (as torch.sort(x2d, dim=-1[, descending=True]) sorts
 * rows).  keys_out[i] is the key of output position i; vals_out[i] is vals_in[j] for the input position j it came from
 * (a gather within the segment), or without vals_in the index j itself -- or j - seg_offsets[s] with
 * LSB_SEG_LOCAL_INDEX, the index within its segment that torch.sort(dim=-1) returns.
 * The contract of lsb_sort_device otherwise: count == here, at least one output, 8-byte aligned device memory of the
 * context's device that is not one of its shards, the caller's stream is waited on, synchronous on return, and with
 * count == 0 no pointer is looked at.  keys_out may alias keys_in; an output must not overlap the other output, vals_in
 * or seg_offsets.  seg_offsets (num_segments + 1 int64) is checked on the device before any key is read: offsets[0] == 0,
 * offsets[num_segments] == count, non-decreasing.  LSB_ERR_ARG for world_size > 1 (one GPU only), num_segments < 1,
 * offsets that fail the check, overlapping outputs, unknown seg_flags, and when the segment id and the input index do
 * not fit one 64-bit word: radix_bits * ceil(bits(num_segments - 1) / radix_bits) + max(1, bits(count - 1)) > 64 (never
 * at radix 16 with count <= 2^32).  Method: the passes of lsb_sort on the keys, then ceil(bits(num_segments - 1) /
 * radix_bits) more on the segment id (uint64 ascending, same pass shape, same skip rule); stats covers the whole call
 * from the pack to the unpack (passes, skipped and subpasses count both kinds).  Afterwards the shard holds internal
 * records: what lsb_download, lsb_checksum and lsb_verify_device report is unspecified until the next sort. */
#define LSB_SEG_LOCAL_INDEX 1u  /* without vals_in: index within the segment instead of the global input index */
int lsb_sort_segments_device(lsb_ctx* ctx, const uint64_t* keys_in, const uint64_t* vals_in, uint64_t* keys_out,
                             uint64_t* vals_out, int64_t count, const int64_t* seg_offsets, int64_t num_segments,
                             uint32_t seg_flags, void* stream, lsb_stats* stats);

/* lsb_sort_device and lsb_sort_segments_device for keys of type key_type (LSB_KEY_*): keys_in and keys_out are arrays
 * of W-bit keys aligned to W / 8 bytes; values and indices stay 8-byte.  With LSB_KEY_CONTEXT they are exactly the two
 * calls above.  A narrow type sorts in ceil(W / radix_bits) key passes (lsb_stats.passes counts them, plus any segment
 * passes), every pass shape and the skip rule as for 8-byte keys.  Contracts as above (multi-GPU: each rank passes its
 * shard; the segmented form is one GPU only), with the pointer and overlap checks on the real byte widths of each
 * array.  LSB_ERR_ARG also for an unknown key_type, a narrow type on a context with LSB_FLAG_KEY_I64 or
 * LSB_FLAG_KEY_F64, and a key pointer not aligned to its width.  After a narrow call the shard holds internal records:
 * what lsb_download, lsb_checksum and lsb_verify_device report is unspecified until the next sort. */
int lsb_sort_device_typed(lsb_ctx* ctx, uint32_t key_type, const void* keys_in, const uint64_t* vals_in, void* keys_out,
                          uint64_t* vals_out, int64_t count, void* stream, lsb_stats* stats);
int lsb_sort_segments_device_typed(lsb_ctx* ctx, uint32_t key_type, const void* keys_in, const uint64_t* vals_in,
                                   void* keys_out, uint64_t* vals_out, int64_t count, const int64_t* seg_offsets,
                                   int64_t num_segments, uint32_t seg_flags, void* stream, lsb_stats* stats);

/* One key column of lsb_lexsort_device.  An 8-byte column has key_type LSB_KEY_CONTEXT and names its type through its
 * own flags (uint64, LSB_FLAG_KEY_I64 or LSB_FLAG_KEY_F64), never through the context's. */
typedef struct lsb_key_column {
  const void* keys;   /* count keys of key_type, device memory aligned to their width                     */
  uint32_t key_type;  /* LSB_KEY_U32 .. LSB_KEY_BF16, or LSB_KEY_CONTEXT: an 8-byte key whose type the
                         column's own flags name (uint64, LSB_FLAG_KEY_I64, LSB_FLAG_KEY_F64)               */
  uint32_t flags;     /* LSB_FLAG_DESCENDING, plus LSB_FLAG_KEY_I64 or LSB_FLAG_KEY_F64 for 8-byte columns    */
} lsb_key_column;

/* Sort by several key columns on device memory, np.lexsort's convention: columns[0] is the least significant key and
 * columns[num_columns - 1] the primary.  The result is the permutation j that sorts stably by
 *   (order_{K-1}(col_{K-1}[j]), ..., order_1(col_1[j]), order_0(col_0[j])),
 * order_c being the key order above of the column's type under its own flags: NaNs last (first when the column is
 * descending), -0.0 == +0.0, a descending column the complement of its order key, and elements equal in every column
 * in input order.  vals_out[i] is vals_in[j[i]], or without vals_in the input index j[i] itself (what np.lexsort
 * returns).  The columns are never rewritten.
 * Method: consecutive columns from columns[0] on share one key word while their widths (64 / 32 / 16 bits) sum to at
 * most 64 and a word holds at most 4 of them; such a round is sorted by ceil(bits / radix_bits) stable passes on its
 * packed order keys (uint64 ascending, the context's pass shape and skip rule), the least significant round first.
 * Each later round repacks the records where they stand, reading its columns at the input index each record carries.
 * So (int32, float32) or (bfloat16, int16, int32) take the 4 passes of one 64-bit sort at radix 16, (int64, int64) two
 * rounds of 4.  stats covers the whole call: passes and skipped count the passes of every round.
 * The contract of lsb_sort_segments_device otherwise: one GPU, count == here, the library's stream waits on `stream`,
 * synchronous on return, and with count == 0 no device pointer is looked at.  Afterwards the shard holds internal
 * records: what lsb_download, lsb_checksum and lsb_verify_device report is unspecified until the next sort.
 * LSB_ERR_ARG, with a message naming the column where one applies, in this order: world_size > 1; a context with
 * LSB_FLAG_KEY_I64, LSB_FLAG_KEY_F64 or LSB_FLAG_DESCENDING (the order comes from the columns only; the pass-shape
 * flags and radix_bits apply as usual); num_columns < 1 or columns == NULL; an unknown key_type; column flags other
 * than LSB_FLAG_DESCENDING (narrow column) or LSB_FLAG_DESCENDING plus one of LSB_FLAG_KEY_I64 / LSB_FLAG_KEY_F64
 * (8-byte column); count != here; and for count > 0: a column with keys == NULL, or not aligned to its width, not
 * device memory of the context's device, or overlapping the context's shards; vals_in failing the same checks at 8
 * bytes; vals_out == NULL or failing them; vals_out overlapping vals_in or any column. */
int lsb_lexsort_device(lsb_ctx* ctx, const lsb_key_column* columns, int32_t num_columns, const uint64_t* vals_in,
                       uint64_t* vals_out, int64_t count, void* stream, lsb_stats* stats);

/* ---- test hooks into the pass (same tables the reference computes) ---------------- */

/* counts[d], d < 2^bits(digit): the localShuffle count loop (:226-229) on this shard; d is the
 * digit of order_key(key) */
int lsb_histogram(lsb_ctx* ctx, int digit, int64_t* host_counts);
/* starts[d]: global output index of the first of MY elements whose digit (of order_key(key)) is d, i.e.
 * GlobalStarts[d*R + myRank] after copyCountsToGlobalCounts + exclusiveScan +
 * copyStartsFromGlobalStarts (:519-525; order defined at :350). Collective. */
int lsb_starts(lsb_ctx* ctx, int digit, int64_t* host_starts);

/* number of passes N_DIGITS = ceil(64/radix_bits) (:22; ceil as chpl:78-79) and the
 * width in bits of digit `digit` (radix_bits, or the remainder for the last one) */
int lsb_num_passes(const lsb_ctx* ctx);
int lsb_digit_bits(const lsb_ctx* ctx, int digit);

/* ---- verification (:710-739, without gathering to rank 0) -------------------------- */

/* order-independent multiset hash of this shard (no communication):
 * out[0] = sum mix(key,val), out[1] = xor mix(key,val), out[2] = xor key, out[3] = sum val */
int lsb_checksum(lsb_ctx* ctx, uint64_t out[4]);

/* Collective.  Checks that (order_key(key),val) is strictly increasing inside every shard and
 * across shard boundaries, and returns the global multiset hash (of the raw key bits).  Because val is the
 * unique original index (:654), "strictly increasing in (key,val) and same multiset as
 * the input" is equivalent to "equals std::stable_sort by key of the input" (:722-726).
 * Returns LSB_ERR_VERIFY if order_violations != 0. */
int lsb_verify_device(lsb_ctx* ctx, lsb_verify* out);

#ifdef __cplusplus
}
#endif
#endif /* LSBSORT_H */
