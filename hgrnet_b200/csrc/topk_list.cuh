// Register-resident sorted top-K list kept by one thread for one image row.
//
// Order: value descending; a new element is inserted only when strictly greater than an
// existing one, so among equal values the element seen first (the lower bank row, because
// every producer streams bank rows in ascending order) stays ahead.  This is the
// deterministic (value desc, index asc) order documented in hgr_b200.h; torch.topk's own
// tie order is unspecified (main.py:138).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace hgr {

// Order key: monotone map fp32 -> uint32 (larger float <=> larger key, -0 below +0) and back.  Lists that leave a
// register or meet in an atomic carry it instead of the float: as the key alone (floor words), or packed into a
// WINNER WORD key << 32 | ~item, whose unsigned order is (value desc, item asc) -- the order above.
__device__ __forceinline__ uint32_t order_key(float v) {
  const uint32_t b = __float_as_uint(v);
  return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}
__device__ __forceinline__ float order_key_value(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
__device__ __forceinline__ unsigned long long winner_word(uint32_t key, uint32_t item) {
  return (static_cast<unsigned long long>(key) << 32) | static_cast<uint32_t>(~item);
}
__device__ __forceinline__ float winner_value(unsigned long long w) {
  return order_key_value(static_cast<uint32_t>(w >> 32));
}
__device__ __forceinline__ int32_t winner_item(unsigned long long w) { return static_cast<int32_t>(~static_cast<uint32_t>(w)); }

template <int KL>
struct SortedList {
  float v[KL];
  int32_t i[KL];

  __device__ __forceinline__ void init() {
#pragma unroll
    for (int j = 0; j < KL; ++j) {
      v[j] = -INFINITY;
      i[j] = -1;
    }
  }
  __device__ __forceinline__ float thr() const { return v[KL - 1]; }

  // pre-condition: x > thr().  Fully unrolled, branch-free (predicated selects).
  __device__ __forceinline__ void insert(float x, int32_t id) {
#pragma unroll
    for (int j = KL - 1; j >= 1; --j) {
      const bool above = x > v[j - 1];  // x lands above slot j-1: slot j inherits slot j-1
      const bool here = x > v[j];       // x lands exactly at slot j
      v[j] = above ? v[j - 1] : (here ? x : v[j]);
      i[j] = above ? i[j - 1] : (here ? id : i[j]);
    }
    if (x > v[0]) {
      v[0] = x;
      i[0] = id;
    }
  }
};

}  // namespace hgr
