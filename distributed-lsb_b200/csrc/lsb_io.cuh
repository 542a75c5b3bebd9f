// lsb_io.cuh -- conversion between a caller's separate key / value arrays on the device (structure of arrays) and the
// shard's 16-byte records (array of structures), for lsb_sort_device.
//
//   pack_kernel<HAS_VALS>     dst[i] = {keys[i], HAS_VALS ? vals[i] : first_global + i}
//   unpack_kernel<KEYS, VALS> keys_out[i] = src[i].key, vals_out[i] = src[i].val (either output may be absent)
//
// Both are pure streams through HBM (bytes per element: pack 24 with the index generated, 32 with vals; unpack 32 with
// both outputs, 24 with one).  A lane touches one element per iteration, so a warp reads 256 contiguous bytes per 8-byte
// array and writes 512 contiguous bytes of records: the caller's arrays need 8-byte alignment only (views such as
// t[1:]), the records are 16-byte aligned in the shard.  U elements per thread are in flight before the first store.
#pragma once
#include "lsb_kernels.cuh"

namespace lsb {

constexpr int IO_THREADS = 256;
constexpr int IO_U = 4;
constexpr int IO_CTAS_PER_SM = 4;  // 1024 threads per SM (all resident at <= 64 registers), U x 16..32 B in flight each

__device__ __forceinline__ uint64_t ld_stream_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}

struct PackArgs {
  const uint64_t* keys;
  const uint64_t* vals;  // HAS_VALS only
  Elt* dst;              // shard buf[0]
  int64_t count;
  int64_t first_global;  // the value of element 0 without vals: its global input index
};

template <bool HAS_VALS>
__global__ void __launch_bounds__(IO_THREADS) pack_kernel(const PackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x;
  for (; i + (IO_U - 1) * stride < a.count; i += IO_U * stride) {
    uint64_t k[IO_U], v[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      k[u] = ld_stream_u64(a.keys + i + u * stride);
      v[u] = HAS_VALS ? ld_stream_u64(a.vals + i + u * stride) : (uint64_t)(a.first_global + i + u * stride);
    }
#pragma unroll
    for (int u = 0; u < IO_U; u++) st_elt(a.dst + i + u * stride, Elt{k[u], v[u]});
  }
  for (; i < a.count; i += stride)
    st_elt(a.dst + i, Elt{ld_stream_u64(a.keys + i), HAS_VALS ? ld_stream_u64(a.vals + i) : (uint64_t)(a.first_global + i)});
}

struct UnpackArgs {
  const Elt* src;  // shard buf[cur] after the sort
  uint64_t* keys;  // KEYS only
  uint64_t* vals;  // VALS only
  int64_t count;
};

template <bool KEYS, bool VALS>
__global__ void __launch_bounds__(IO_THREADS) unpack_kernel(const UnpackArgs a) {
  const int64_t stride = (int64_t)gridDim.x * IO_THREADS;
  int64_t i = (int64_t)blockIdx.x * IO_THREADS + threadIdx.x;
  for (; i + (IO_U - 1) * stride < a.count; i += IO_U * stride) {
    Elt e[IO_U];
#pragma unroll
    for (int u = 0; u < IO_U; u++) e[u] = ld_stream(a.src + i + u * stride);
#pragma unroll
    for (int u = 0; u < IO_U; u++) {
      if (KEYS) a.keys[i + u * stride] = e[u].key;
      if (VALS) a.vals[i + u * stride] = e[u].val;
    }
  }
  for (; i < a.count; i += stride) {
    const Elt e = ld_stream(a.src + i);
    if (KEYS) a.keys[i] = e.key;
    if (VALS) a.vals[i] = e.val;
  }
}

}  // namespace lsb
