// lsb_io.cuh -- conversion between a caller's separate key / value arrays on the device (structure of arrays) and the
// shard's 16-byte records (array of structures), for lsb_sort_device and lsb_sort_device_typed.
//
//   pack_kernel<KT, HAS_VALS>         dst[i] = {key_word(keys[i]), HAS_VALS ? vals[i] : first_global + i}
//   unpack_kernel<KBYTES, KEYS, VALS> keys_out[i] = key of src[i].key, vals_out[i] = src[i].val (either may be absent)
//
// KT is an LSB_KEY_* type: LSB_KEY_CONTEXT moves the 8-byte key as it is; a narrow type reads a W-bit key and packs
// narrow_key_word (lsb_keyorder.cuh), and the unpack of KBYTES = W / 8 writes the word's high half back.
// Both are pure streams through HBM (bytes per element: pack 16 + KBYTES with the index generated, 24 + KBYTES with
// vals; unpack 16 + KBYTES + 8 with both outputs).  A lane touches one element per iteration, so the caller's arrays need
// alignment to their own element width only (views such as t[1:]); the records are 16-byte aligned in the shard.  U
// elements per thread are in flight before the first store.
#pragma once
#include "lsb_kernels.cuh"
#include "lsb_keyorder.cuh"

namespace lsb {

constexpr int IO_THREADS = 256;
constexpr int IO_U = 4;
constexpr int IO_CTAS_PER_SM = 4;  // 1024 threads per SM (all resident at <= 64 registers), U x 16..32 B in flight each

__device__ __forceinline__ uint64_t ld_stream_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t ld_stream_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t ld_stream_u16(const uint16_t* p) {
  unsigned short v;
  asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return v;
}

// key word of input key i of type KT (flags: the context's, for a narrow key's DESCENDING)
template <int KT>
__device__ __forceinline__ uint64_t ld_key_word(const void* keys, int64_t i, uint32_t flags) {
  if (KT == LSB_KEY_CONTEXT) return ld_stream_u64((const uint64_t*)keys + i);
  const uint32_t k = key_type_bits(KT) == 32 ? ld_stream_u32((const uint32_t*)keys + i) : ld_stream_u16((const uint16_t*)keys + i);
  return narrow_key_word(k, KT, flags);
}

// keys_out[i] from a record's key word: the word itself (8 bytes) or its high half at KBYTES = 4 / 2
template <int KBYTES>
__device__ __forceinline__ void st_key(void* keys, int64_t i, uint64_t word) {
  if (KBYTES == 8) ((uint64_t*)keys)[i] = word;
  else if (KBYTES == 4) ((uint32_t*)keys)[i] = (uint32_t)(word >> 32);
  else ((uint16_t*)keys)[i] = (uint16_t)(word >> 32);
}

struct PackArgs {
  const void* keys;
  const uint64_t* vals;  // HAS_VALS only
  Elt* dst;              // shard buf[0]
  int64_t count;
  int64_t first_global;  // the value of element 0 without vals: its global input index
  uint32_t flags;        // narrow KT: the key order (DESCENDING) applied to the key word
};

template <int KT, bool HAS_VALS>
__global__ void __launch_bounds__(IO_THREADS) pack_kernel(const PackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x;
  for (; i + (IO_U - 1) * stride < a.count; i += IO_U * stride) {
    uint64_t k[IO_U], v[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      k[u] = ld_key_word<KT>(a.keys, i + u * stride, a.flags);
      v[u] = HAS_VALS ? ld_stream_u64(a.vals + i + u * stride) : (uint64_t)(a.first_global + i + u * stride);
    }
#pragma unroll
    for (int u = 0; u < IO_U; u++) st_elt(a.dst + i + u * stride, Elt{k[u], v[u]});
  }
  for (; i < a.count; i += stride)
    st_elt(a.dst + i, Elt{ld_key_word<KT>(a.keys, i, a.flags), HAS_VALS ? ld_stream_u64(a.vals + i) : (uint64_t)(a.first_global + i)});
}

struct UnpackArgs {
  const Elt* src;  // shard buf[cur] after the sort
  void* keys;      // KEYS only
  uint64_t* vals;  // VALS only
  int64_t count;
};

template <int KBYTES, bool KEYS, bool VALS>
__global__ void __launch_bounds__(IO_THREADS) unpack_kernel(const UnpackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x;
  for (; i + (IO_U - 1) * stride < a.count; i += IO_U * stride) {
    Elt e[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) e[u] = ld_stream(a.src + i + u * stride);
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      if (KEYS) st_key<KBYTES>(a.keys, i + u * stride, e[u].key);
      if (VALS) a.vals[i + u * stride] = e[u].val;
    }
  }
  for (; i < a.count; i += stride) {
    const Elt e = ld_stream(a.src + i);
    if (KEYS) st_key<KBYTES>(a.keys, i, e.key);
    if (VALS) a.vals[i] = e.val;
  }
}

}  // namespace lsb
