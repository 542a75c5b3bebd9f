// lsb_keyorder.cuh -- the key orders of include/lsbsort.h (LSB_FLAG_KEY_I64, LSB_FLAG_KEY_F64,
// LSB_FLAG_DESCENDING) in one place.  A sort under `flags` is the stable sort ascending by
// order_key(key, flags); every kernel that reads a digit reads it from order_key of the key it holds,
// and the host's cross-shard check compares order_key too.  The key bits themselves are never
// rewritten: -0.0 stays -0.0 and a NaN keeps its sign and payload.  The narrow key types (LSB_KEY_U32 .. LSB_KEY_BF16)
// apply the same rules at their own width in the pack (order_key_narrow); their passes then read the key word as a
// uint64 ascending.
#pragma once
#include <stdint.h>

#include "../../include/lsbsort.h"

namespace lsb {

// uint64: k.  int64: k ^ 2^63.  float64: -0.0 as +0.0 (they compare equal), every NaN (either sign, any
// payload) as ~0 (last), any other value k ^ (sign ? ~0 : 2^63).  DESCENDING: the complement of that.
// These are the orders of np.argsort(kind="stable") and torch.sort(stable=True[, descending=True]).
__host__ __device__ __forceinline__ uint64_t order_key(uint64_t k, uint32_t flags) {
  if (flags & LSB_FLAG_KEY_F64) {
    if ((k << 1) == 0) k = 0;
    k = (k << 1) > (0x7FFULL << 53) ? ~0ULL : k ^ ((uint64_t)((int64_t)k >> 63) | (1ULL << 63));
  } else if (flags & LSB_FLAG_KEY_I64) {
    k ^= 1ULL << 63;
  }
  return (flags & LSB_FLAG_DESCENDING) ? ~k : k;
}

// Key width in bits of an LSB_KEY_* type: 64 for LSB_KEY_CONTEXT, 32 or 16 for the narrow types, 0 for an unknown one.
__host__ __device__ __forceinline__ int key_type_bits(uint32_t key_type) {
  return key_type == LSB_KEY_CONTEXT ? 64 : key_type <= LSB_KEY_F32 ? 32 : key_type <= LSB_KEY_BF16 ? 16 : 0;
}

// The W-bit order key of a narrow key k (W = key_type_bits(key_type), k in the low W bits), the rule of order_key at
// width W.  uint: k.  int: k ^ signbit.  float32 / float16 / bfloat16: -0 as +0, every NaN ((k << 1) > (inf << 1) in W
// bits, either sign, any payload) as all ones, any other value k ^ (sign ? all ones : signbit).  DESCENDING: the
// complement within W bits.
__host__ __device__ __forceinline__ uint32_t order_key_narrow(uint32_t k, uint32_t key_type, uint32_t flags) {
  const uint32_t all = key_type_bits(key_type) == 32 ? 0xFFFFFFFFu : 0xFFFFu, sign = all ^ (all >> 1);
  k &= all;
  if (key_type == LSB_KEY_I32 || key_type == LSB_KEY_I16) {
    k ^= sign;
  } else if (key_type == LSB_KEY_F32 || key_type == LSB_KEY_F16 || key_type == LSB_KEY_BF16) {
    const uint32_t inf = key_type == LSB_KEY_F32 ? 0x7F800000u : key_type == LSB_KEY_F16 ? 0x7C00u : 0x7F80u;
    const uint32_t mag = (k << 1) & all;
    if (mag == 0) k = 0;
    k = mag > ((inf << 1) & all) ? all : k ^ ((k & sign) ? all : sign);
  }
  return (flags & LSB_FLAG_DESCENDING) ? ~k & all : k;
}

// The key word of a narrow key's record: the raw bits above, the order key in the low W bits.  The passes sort the low
// W bits only; the unpack writes key_word >> 32 back at width W, so the key bits are never rewritten.
__host__ __device__ __forceinline__ uint64_t narrow_key_word(uint32_t k, uint32_t key_type, uint32_t flags) {
  return (uint64_t)k << 32 | order_key_narrow(k, key_type, flags);
}

}  // namespace lsb
