// Warp-level exact scan of one image row against a range of bank rows on the CUDA cores.
// Shared by the SIMT implementation (score_simt.cu) and by the exactness fallback of the merge
// kernel (topk_merge.cu): the list is replicated in every lane (all lanes see the same sums).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "topk_list.cuh"

namespace hgr {

__device__ __forceinline__ float dot8_bf16(const uint4& a, const uint4& b, float acc) {
  const uint32_t ua[4] = {a.x, a.y, a.z, a.w};
  const uint32_t ub[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    acc = fmaf(__uint_as_float(ua[i] << 16), __uint_as_float(ub[i] << 16), acc);
    acc = fmaf(__uint_as_float(ua[i] & 0xFFFF0000u), __uint_as_float(ub[i] & 0xFFFF0000u), acc);
  }
  return acc;
}

__device__ __forceinline__ float warp_sum_f32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float warp_max_f32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// xr: the image row as D8 uint4 (8 bf16 each), readable by every lane (shared or global memory).
template <int KL>
__device__ __forceinline__ void scan_row_range(const uint4* xr, const uint4* __restrict__ bank4, int64_t c0,
                                               int64_t c1, int D8, int lane, SortedList<KL>& list) {
  int64_t c = c0;
  for (; c + 1 < c1; c += 2) {
    float a0 = 0.f, a1 = 0.f;
    const uint4* b0 = bank4 + c * D8;
    const uint4* b1 = b0 + D8;
    for (int idx = lane; idx < D8; idx += 32) {
      const uint4 x = xr[idx];
      a0 = dot8_bf16(__ldg(b0 + idx), x, a0);
      a1 = dot8_bf16(__ldg(b1 + idx), x, a1);
    }
    a0 = warp_sum_f32(a0);
    a1 = warp_sum_f32(a1);
    if (a0 > list.thr()) list.insert(a0, static_cast<int32_t>(c));
    if (a1 > list.thr()) list.insert(a1, static_cast<int32_t>(c + 1));
  }
  if (c < c1) {
    float a0 = 0.f;
    const uint4* b0 = bank4 + c * D8;
    for (int idx = lane; idx < D8; idx += 32) a0 = dot8_bf16(__ldg(b0 + idx), xr[idx], a0);
    a0 = warp_sum_f32(a0);
    if (a0 > list.thr()) list.insert(a0, static_cast<int32_t>(c));
  }
}

// Same result set, organised for a LONE warp (the exact repair in the merge kernel): every lane owns one bank row
// of a 32-row block and streams it sequentially (its 128-byte lines are re-used from L1 over eight loads, 32
// independent rows in flight), the image row is a warp-uniform broadcast load, and the 32 finished dot products
// are offered to the replicated list in ascending row order.  ~10x the throughput of scan_row_range for one warp,
// which waits a full memory round trip for every two rows.
// `rows` (optional) keeps only the bank rows c with rows(c) true, tested before the row's operands are loaded; the
// default takes every row and loads unconditionally (a lane past c1 re-reads row c0).
struct EveryRow {
  static constexpr bool kFilter = false;
  __device__ __forceinline__ bool operator()(int64_t) const { return true; }
};

template <int KL, class Rows = EveryRow>
__device__ __forceinline__ void scan_row_range_lanes(const uint4* __restrict__ xr, const uint4* __restrict__ bank4,
                                                     int64_t c0, int64_t c1, int D8, int lane, SortedList<KL>& list,
                                                     const Rows& rows = Rows()) {
  for (int64_t cb = c0; cb < c1; cb += 32) {
    const int64_t c = cb + lane;
    const bool ok = c < c1 && rows(c);
    const uint4* b = bank4 + (ok ? c : c0) * D8;
    float a0 = 0.f, a1 = 0.f;
    if (ok || !Rows::kFilter) {
      int idx = 0;
      for (; idx + 1 < D8; idx += 2) {
        const uint4 x0 = __ldg(xr + idx), x1 = __ldg(xr + idx + 1);
        a0 = dot8_bf16(__ldg(b + idx), x0, a0);
        a1 = dot8_bf16(__ldg(b + idx + 1), x1, a1);
      }
      if (idx < D8) a0 = dot8_bf16(__ldg(b + idx), __ldg(xr + idx), a0);
    }
    const float v = ok ? a0 + a1 : -INFINITY;
    if (warp_max_f32(v) > list.thr()) {
      for (int l = 0; l < 32; ++l) {
        const float vl = __shfl_sync(0xffffffffu, v, l);
        if (vl > list.thr()) list.insert(vl, static_cast<int32_t>(cb + l));
      }
    }
  }
}

}  // namespace hgr
