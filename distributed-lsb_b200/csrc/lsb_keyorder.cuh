// lsb_keyorder.cuh -- the key orders of include/lsbsort.h (LSB_FLAG_KEY_I64, LSB_FLAG_KEY_F64,
// LSB_FLAG_DESCENDING) in one place.  A sort under `flags` is the stable sort ascending by
// order_key(key, flags); every kernel that reads a digit reads it from order_key of the key it holds,
// and the host's cross-shard check compares order_key too.  The key bits themselves are never
// rewritten: -0.0 stays -0.0 and a NaN keeps its sign and payload.
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

}  // namespace lsb
