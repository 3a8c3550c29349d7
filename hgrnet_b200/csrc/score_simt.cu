// CUDA-core implementation of the scoring head (HGR_IMPL_SIMT).
//
// Same contract as the tcgen05 kernel (score_pair.cu): logits = X @ bank^T, per-row sorted
// top-K, never materialising B x C.  It accepts any shape (D % 8 == 0) and exists for three
// reasons: (a) shapes the tensor-core kernel does not take, (b) an on-device cross-check of
// the tcgen05 path in the GPU tests, (c) its row scan (simt_row.cuh) is the exact re-scan of
// rows whose speculative narrow lists could not be certified (topk_merge.cu).  It is NOT a
// CPU fallback.
//
// Reference: model/clip_tree.py:331 (`feats @ self.zsl_weights.T`) + main.py:136-141.
#include "common.cuh"
#include "sched.cuh"
#include "simt_row.cuh"

namespace hgr {
namespace {

constexpr int kSimtWarps = 8;

__device__ __forceinline__ void stage_rows(uint4* s_x, const uint4* X4, int64_t B, int D8) {
  for (int i = threadIdx.x; i < kSimtWarps * D8; i += blockDim.x) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * kSimtWarps + i / D8;
    s_x[i] = r < B ? X4[r * D8 + i % D8] : make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
}

template <int KL>
__global__ void __launch_bounds__(kSimtWarps * 32)
score_topk_simt_kernel(const uint4* __restrict__ X4, const uint4* __restrict__ bank4, int64_t B, int64_t C,
                       int D8, int64_t cols_per_split, int K, float* __restrict__ part_val,
                       int32_t* __restrict__ part_idx) {
  extern __shared__ uint4 s_x[];
  stage_rows(s_x, X4, B, D8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kSimtWarps + warp;
  if (row >= B) return;
  const int64_t c0 = blockIdx.y * cols_per_split;
  const int64_t c1 = c0 + cols_per_split < C ? c0 + cols_per_split : C;
  SortedList<KL> list;
  list.init();
  scan_row_range<KL>(s_x + warp * D8, bank4, c0, c1, D8, lane, list);
  if (lane == 0) {
    float* pv = part_val + (static_cast<int64_t>(blockIdx.y) * B + row) * K;
    int32_t* pi = part_idx + (static_cast<int64_t>(blockIdx.y) * B + row) * K;
#pragma unroll
    for (int k = 0; k < KL; ++k) {
      if (k < K) {
        pv[k] = list.v[k];
        pi[k] = list.i[k];
      }
    }
  }
}

__global__ void __launch_bounds__(kSimtWarps * 32)
logits_simt_kernel(const uint4* __restrict__ X4, const uint4* __restrict__ bank4, int64_t B, int64_t C, int D8,
                   int64_t cols_per_split, float scale, float* __restrict__ out, int64_t ldo) {
  extern __shared__ uint4 s_x[];
  stage_rows(s_x, X4, B, D8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kSimtWarps + warp;
  if (row >= B) return;
  const int64_t c0 = blockIdx.y * cols_per_split;
  const int64_t c1 = c0 + cols_per_split < C ? c0 + cols_per_split : C;
  const uint4* xr = s_x + warp * D8;
  for (int64_t cb = c0; cb < c1; cb += 32) {
    float keep = 0.f;
    for (int j = 0; j < 32 && cb + j < c1; ++j) {
      float a = 0.f;
      const uint4* b = bank4 + (cb + j) * D8;
      for (int idx = lane; idx < D8; idx += 32) a = dot8_bf16(__ldg(b + idx), xr[idx], a);
      a = warp_sum_f32(a);
      if (lane == j) keep = a;
    }
    if (cb + lane < c1) out[row * ldo + cb + lane] = keep * scale;
  }
}

int pick_splits(int64_t B, int64_t C) {
  const int64_t row_blocks = (B + kSimtWarps - 1) / kSimtWarps;
  int64_t s = (4LL * num_sms() + row_blocks - 1) / row_blocks;
  const int64_t max_by_cols = (C + 63) / 64;
  if (s > max_by_cols) s = max_by_cols;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  return static_cast<int>(s);
}

}  // namespace

// The partial lists sit behind the header of the scoring workspace, which carries the tcgen05 calls' state between
// calls (umma_common.cuh: re-scan count, floor-sketch epoch) and is left alone here.
size_t simt_score_workspace_bytes(int64_t B, int64_t C, int K) {
  return static_cast<size_t>(pick_splits(B, C)) * B * K * (sizeof(float) + sizeof(int32_t)) + kScoreWsHeaderBytes;
}

int launch_score_topk_simt(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                           int32_t id_base, const int32_t* targets, int64_t B, int64_t C, int64_t D, float scale,
                           int K, void* ws, size_t ws_bytes, float* topk_val, int32_t* topk_idx, int64_t* hits,
                           cudaStream_t stream, const OutScatter* scatter) {
  const int S = pick_splits(B, C);
  const size_t need = simt_score_workspace_bytes(B, C, K);
  if (ws_bytes < need || ws == nullptr)
    return set_error(HGR_ERR_WORKSPACE, "hgr_score_topk(simt): workspace %zu < %zu bytes", ws_bytes, need);
  float* part_val = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + kScoreWsHeaderBytes);
  int32_t* part_idx = reinterpret_cast<int32_t*>(part_val + static_cast<size_t>(S) * B * K);
  const int D8 = static_cast<int>(D / 8);
  const size_t smem = static_cast<size_t>(kSimtWarps) * D8 * sizeof(uint4);
  const int64_t cps = (C + S - 1) / S;
  dim3 grid(static_cast<unsigned>((B + kSimtWarps - 1) / kSimtWarps), S);
  if (smem > 200 * 1024) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk(simt): D = %lld too large", (long long)D);
#define HGR_SIMT_LAUNCH(KL)                                                                                      \
  do {                                                                                                           \
    if (smem > 48 * 1024)                                                                                        \
      HGR_CHECK_CUDA(cudaFuncSetAttribute(score_topk_simt_kernel<KL>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                          static_cast<int>(smem)));                                              \
    score_topk_simt_kernel<KL><<<grid, kSimtWarps * 32, smem, stream>>>(                                         \
        reinterpret_cast<const uint4*>(X), reinterpret_cast<const uint4*>(bank), B, C, D8, cps, K, part_val,     \
        part_idx);                                                                                               \
  } while (0)
  if (K <= 8) HGR_SIMT_LAUNCH(8);
  else if (K <= 20) HGR_SIMT_LAUNCH(20);
  else HGR_SIMT_LAUNCH(32);
#undef HGR_SIMT_LAUNCH
  HGR_CHECK_LAUNCH();
  MergeArgs m{};
  m.part_val = part_val;
  m.part_idx = part_idx;
  m.P = S;
  m.B = B;
  m.KL = K;
  m.K = K;
  m.col_id = col_id;
  m.id_base = id_base;
  m.scale = scale;
  m.targets = targets;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  m.hits = hits;
  if (scatter) m.scatter = *scatter;
  return launch_topk_merge(m, stream);
}

int launch_logits_simt(const __nv_bfloat16* X, const __nv_bfloat16* bank, int64_t B, int64_t C, int64_t D,
                       float scale, float* out, int64_t ldo, cudaStream_t stream) {
  const int S = pick_splits(B, C);
  const int D8 = static_cast<int>(D / 8);
  const size_t smem = static_cast<size_t>(kSimtWarps) * D8 * sizeof(uint4);
  if (smem > 200 * 1024) return set_error(HGR_ERR_UNSUPPORTED, "hgr_logits_dense(simt): D = %lld too large", (long long)D);
  if (smem > 48 * 1024)
    HGR_CHECK_CUDA(cudaFuncSetAttribute(logits_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
  int64_t cps = (C + S - 1) / S;
  cps = (cps + 31) / 32 * 32;
  dim3 grid(static_cast<unsigned>((B + kSimtWarps - 1) / kSimtWarps), S);
  logits_simt_kernel<<<grid, kSimtWarps * 32, smem, stream>>>(reinterpret_cast<const uint4*>(X),
                                                              reinterpret_cast<const uint4*>(bank), B, C, D8, cps,
                                                              scale, out, ldo);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
