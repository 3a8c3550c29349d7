// extern "C" surface of libhgr_b200.so (declared in include/hgr_b200.h): argument checks,
// implementation selection and error reporting.  No device memory is allocated here.
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "sched.cuh"

namespace hgr {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int num_sms() {
  static int cached = [] {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      return kNumSMsB200;  // no device visible (build box): size queries assume a B200
    }
    return n;
  }();
  return cached;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int pick_impl(int impl, int64_t B, int64_t C, int64_t D, int K) {
  if (impl == HGR_IMPL_AUTO) {
    const char* e = getenv("HGR_IMPL");
    if (e && !strcmp(e, "simt")) return HGR_IMPL_SIMT;
    return umma_supported(B, C, D, K) ? HGR_IMPL_TCGEN05 : HGR_IMPL_SIMT;
  }
  return impl;
}

}  // namespace hgr

using namespace hgr;

extern "C" {

int hgr_version(void) { return HGR_ABI_VERSION; }

const char* hgr_last_error(void) { return g_err; }

int64_t hgr_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int hgr_aggregate_normalize(const void* E, int e_dtype, int64_t n_src, int64_t D, const int32_t* rowptr,
                            const int32_t* col, const float* w, int64_t n_rows, const int32_t* row_map,
                            int64_t n_out, void* out, int out_dtype, float* out_norm, void* stream) {
  HGR_CHECK_ARG(n_src >= 0 && n_rows >= 0 && n_out >= 0, "hgr_aggregate_normalize: negative size");
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_aggregate_normalize: D = %lld must be a positive multiple of 8", (long long)D);
  if (n_out == 0) return HGR_OK;
  HGR_CHECK_ARG(E && out, "hgr_aggregate_normalize: null E/out");
  HGR_CHECK_ARG(aligned16(E) && aligned16(out), "hgr_aggregate_normalize: E/out must be 16-byte aligned");
  HGR_CHECK_ARG(rowptr == nullptr || col != nullptr, "hgr_aggregate_normalize: rowptr given without col");
  HGR_CHECK_ARG(rowptr != nullptr || n_rows == n_src, "hgr_aggregate_normalize: identity CSR needs n_rows == n_src");
  HGR_CHECK_ARG(row_map != nullptr || n_out == n_rows, "hgr_aggregate_normalize: n_out != n_rows without row_map");
  HGR_CHECK_ARG(n_src < (int64_t(1) << 31) && n_rows < (int64_t(1) << 31), "hgr_aggregate_normalize: > 2^31 rows");
  return launch_aggregate_normalize(E, e_dtype, n_src, D, rowptr, col, w, row_map, n_out, out, out_dtype, out_norm,
                                    static_cast<cudaStream_t>(stream));
}

int hgr_normalize_rows_dual(const void* E, int e_dtype, int64_t n_rows, int64_t D, void* out, const int32_t* dst_map,
                            void* out2, void* stream) {
  HGR_CHECK_ARG(n_rows >= 0, "hgr_normalize_rows_dual: negative size");
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_normalize_rows_dual: D = %lld must be a positive multiple of 8", (long long)D);
  if (n_rows == 0) return HGR_OK;
  HGR_CHECK_ARG(E && out, "hgr_normalize_rows_dual: null E/out");
  HGR_CHECK_ARG((dst_map == nullptr) == (out2 == nullptr), "hgr_normalize_rows_dual: dst_map and out2 go together");
  HGR_CHECK_ARG(aligned16(E) && aligned16(out) && aligned16(out2), "hgr_normalize_rows_dual: E/out/out2 must be 16-byte aligned");
  return launch_normalize_dual(E, e_dtype, n_rows, D, out, dst_map, out2, static_cast<cudaStream_t>(stream));
}

size_t hgr_score_topk_workspace_bytes(int64_t B, int64_t C, int64_t D, int K) {
  if (B <= 0 || C <= 0 || K <= 0) return 16;
  size_t a = simt_score_workspace_bytes(B, C, K);
  size_t b = umma_supported(B, C, D, K) ? umma_score_workspace_bytes(B, C, K) : 0;
  return (a > b ? a : b) + 16;
}

// The merge of zero lists: every row gets (-inf, -1) -- and, scattered with bounds, a -inf bound.
static int merge_zero_lists(int64_t B, int K, float* topk_val, int32_t* topk_idx, const OutScatter* scatter,
                            cudaStream_t stream) {
  MergeArgs m{};
  m.B = B;
  m.KL = K;
  m.K = K;
  m.scale = 1.f;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  if (scatter) m.scatter = *scatter;
  return launch_topk_merge(m, stream);
}

static int score_topk_impl(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, const int32_t* targets,
                           int64_t B, int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                           float* topk_val, int32_t* topk_idx, int64_t* hits, int impl, void* stream,
                           const OutScatter* scatter, int64_t C_total = 0) {
  HGR_CHECK_ARG(B >= 0 && C >= 0, "hgr_score_topk: negative size");
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_score_topk: D = %lld must be a positive multiple of 8", (long long)D);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(scale > 0.f, "hgr_score_topk: scale must be > 0 (top-k order is taken on unscaled cosines)");
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(scatter || (topk_val && topk_idx), "hgr_score_topk: null output");
  HGR_CHECK_ARG(C == 0 || (X && bank), "hgr_score_topk: null X/bank");
  HGR_CHECK_ARG(aligned16(X) && aligned16(bank) && aligned16(workspace), "hgr_score_topk: X/bank/workspace must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (C == 0) return merge_zero_lists(B, K, topk_val, topk_idx, scatter, s);   // empty class set
  const bool skip_merge = (impl & HGR_IMPL_FLAG_NO_MERGE) != 0;
  const int share = (impl & HGR_IMPL_GRID_SHARE_MASK) >> HGR_IMPL_GRID_SHARE_SHIFT;
  HGR_CHECK_ARG(share <= HGR_GRID_SHARE_MAX, "hgr_score_topk: grid share %d outside [0, %d]", share, HGR_GRID_SHARE_MAX);
  impl &= ~(HGR_IMPL_FLAG_NO_MERGE | HGR_IMPL_GRID_SHARE_MASK);
  const int which = pick_impl(impl, B, C, D, K);
  if (which == HGR_IMPL_TCGEN05 || which == HGR_IMPL_TCGEN05_EXACT || which == HGR_IMPL_TCGEN05_NULL ||
      which == HGR_IMPL_TCGEN05_SKETCH) {
    if (!umma_supported(B, C, D, K)) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk: shape not supported by the tcgen05 kernel");
    const int variant = which - HGR_IMPL_TCGEN05;  // umma::Variant
    return launch_score_topk_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), col_id,
                                  id_base, targets, B, C, D, scale, K, workspace, workspace_bytes, topk_val, topk_idx,
                                  hits, variant, skip_merge || which == HGR_IMPL_TCGEN05_NULL, s, scatter, C_total,
                                  share > 1 ? share : 1);
  }
  if (which == HGR_IMPL_SIMT)
    return launch_score_topk_simt(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), col_id,
                                  id_base, targets, B, C, D, scale, K, workspace, workspace_bytes, topk_val, topk_idx,
                                  hits, s, scatter);
  return set_error(HGR_ERR_BAD_ARG, "hgr_score_topk: unknown impl %d", impl);
}

// main.py:104-222 run once per split (`--model_test` / `--data_test` = 2-hops, 3-hops, all): one GEMM over the union
// bank, per split the top-K of main.py:136-138 and the hit / row counts of main.py:139-147.
static int split_table(int64_t C, int n_groups, const int32_t* group_end, const uint8_t* group_splits, int n_splits,
                       Groups* gr) {
  HGR_CHECK_ARG(n_splits >= 1 && n_splits <= kMaxSplits, "hgr_score_topk_splits: %d splits outside [1, %d]", n_splits,
                kMaxSplits);
  HGR_CHECK_ARG(group_end != nullptr && group_splits != nullptr, "hgr_score_topk_splits: null group table");
  HGR_CHECK_ARG(make_groups(C, n_groups, group_end, gr),
                "hgr_score_topk_splits: %d groups: need 1..%d strictly ascending ends, the last = C = %lld", n_groups,
                kMaxGroups, (long long)C);
  for (int g = 0; g < n_groups; ++g)
    HGR_CHECK_ARG(group_splits[g] < (1u << n_splits), "hgr_score_topk_splits: group %d names a split >= %d", g, n_splits);
  return HGR_OK;
}

size_t hgr_score_topk_splits_workspace_bytes(int64_t B, int64_t C, int64_t D, int K, int n_groups, const int32_t* group_end) {
  Groups gr;
  if (B <= 0 || C <= 0 || K <= 0 || K > HGR_TOPK_MAX || group_end == nullptr || !make_groups(C, n_groups, group_end, &gr))
    return 16;
  return umma_split_workspace_bytes(B, gr, K) + 16;
}

int hgr_score_topk_splits(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, const int32_t* targets,
                          const uint8_t* node_splits, int64_t n_nodes, int64_t B, int64_t C, int64_t D, float scale, int K,
                          int n_groups, const int32_t* group_end, const uint8_t* group_splits, int n_splits,
                          void* workspace, size_t workspace_bytes, float* topk_val, int32_t* topk_idx, int64_t* counts,
                          int impl, void* stream) {
  HGR_CHECK_ARG(B >= 0 && C >= 1, "hgr_score_topk_splits: bad sizes B=%lld C=%lld", (long long)B, (long long)C);
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_score_topk_splits: D = %lld must be a positive multiple of 8", (long long)D);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_splits: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(scale > 0.f, "hgr_score_topk_splits: scale must be > 0 (top-k order is taken on unscaled cosines)");
  Groups gr;
  const int rc = split_table(C, n_groups, group_end, group_splits, n_splits, &gr);
  if (rc != HGR_OK) return rc;
  if (impl != HGR_IMPL_AUTO && impl != HGR_IMPL_TCGEN05 && impl != HGR_IMPL_TCGEN05_EXACT)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_splits: impl %d (only the tcgen05 kernel has the grouped schedule)",
                     impl);
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(X && bank && topk_val && topk_idx, "hgr_score_topk_splits: null X / bank / output");
  HGR_CHECK_ARG(counts == nullptr || (targets && node_splits && n_nodes > 0),
                "hgr_score_topk_splits: counting needs targets and node_splits");
  HGR_CHECK_ARG(aligned16(X) && aligned16(bank) && aligned16(workspace), "hgr_score_topk_splits: X/bank/workspace must be 16-byte aligned");
  if (!umma_supported(B, C, D, K)) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_splits: shape not supported by the tcgen05 kernel");
  return launch_score_topk_splits_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), col_id,
                                       id_base, counts ? targets : nullptr, node_splits, n_nodes, B, C, D, scale, K, gr,
                                       group_splits, n_splits, workspace, workspace_bytes, topk_val, topk_idx, counts,
                                       impl == HGR_IMPL_TCGEN05_EXACT, static_cast<cudaStream_t>(stream));
}

// Class shard of the union bank, one rank's part of main.py:104-222 run once per split: per split the rank's top-K and
// the bound of what it dropped, scattered to the row owners (hgr_topk_merge_splits_certified).
static int split_totals(int n_splits, const int64_t* split_C_total) {
  HGR_CHECK_ARG(split_C_total != nullptr, "hgr_score_topk_splits_scatter_bounded: null split_C_total");
  for (int sp = 0; sp < n_splits; ++sp)
    HGR_CHECK_ARG(split_C_total[sp] >= 0, "hgr_score_topk_splits_scatter_bounded: split_C_total[%d] = %lld < 0", sp,
                  (long long)split_C_total[sp]);
  return HGR_OK;
}

size_t hgr_score_topk_splits_scatter_bounded_workspace_bytes(int64_t B, int64_t C, int64_t D, int K, int n_groups,
                                                             const int32_t* group_end) {
  return hgr_score_topk_splits_workspace_bytes(B, C, D, K, n_groups, group_end);
}

int hgr_score_topk_splits_scatter_bounded(const void* X, const void* bank, const int32_t* col_id, int32_t id_base,
                                          int64_t B, int64_t C, int64_t D, float scale, int K, int n_groups,
                                          const int32_t* group_end, const uint8_t* group_splits, int n_splits,
                                          const int64_t* split_C_total, void* workspace, size_t workspace_bytes,
                                          int64_t block_rows, int n_blocks, float* const* val_blocks,
                                          int32_t* const* idx_blocks, float* const* bound_blocks, int64_t split_stride,
                                          int impl, void* stream) {
  HGR_CHECK_ARG(B >= 0 && C >= 0, "hgr_score_topk_splits_scatter_bounded: bad sizes B=%lld C=%lld", (long long)B,
                (long long)C);
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_score_topk_splits_scatter_bounded: D = %lld must be a positive multiple of 8",
                (long long)D);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_splits_scatter_bounded: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(scale > 0.f, "hgr_score_topk_splits_scatter_bounded: scale must be > 0");
  HGR_CHECK_ARG(n_splits >= 1 && n_splits <= kMaxSplits, "hgr_score_topk_splits_scatter_bounded: %d splits outside [1, %d]",
                n_splits, kMaxSplits);
  Groups gr;
  if (C > 0) {
    const int rc = split_table(C, n_groups, group_end, group_splits, n_splits, &gr);
    if (rc != HGR_OK) return rc;
  }
  int rc = split_totals(n_splits, split_C_total);
  if (rc != HGR_OK) return rc;
  if (impl != HGR_IMPL_AUTO && impl != HGR_IMPL_TCGEN05)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_splits_scatter_bounded: impl %d (only the tcgen05 kernel has the "
                     "grouped schedule)", impl);
  HGR_CHECK_ARG(n_blocks >= 1 && n_blocks <= kMaxScatterBlocks,
                "hgr_score_topk_splits_scatter_bounded: n_blocks = %d outside [1, %d]", n_blocks, kMaxScatterBlocks);
  HGR_CHECK_ARG(block_rows >= 1 && block_rows * n_blocks >= B,
                "hgr_score_topk_splits_scatter_bounded: %d blocks of %lld rows do not cover B = %lld", n_blocks,
                (long long)block_rows, (long long)B);
  HGR_CHECK_ARG(val_blocks && idx_blocks && bound_blocks, "hgr_score_topk_splits_scatter_bounded: null block tables");
  // a split's area in an owner's slot: the value and id lists [n_blocks, block_rows, K] and the bounds [n_blocks,
  // block_rows] of all producers
  HGR_CHECK_ARG(n_splits == 1 || split_stride >= n_blocks * block_rows * (2 * K + 1),
                "hgr_score_topk_splits_scatter_bounded: split_stride %lld < %lld: the areas of two splits overlap",
                (long long)split_stride, (long long)(n_blocks * block_rows * (2 * K + 1)));
  if (B == 0) return HGR_OK;
  OutScatter sc;
  sc.n_blocks = n_blocks;
  sc.block_rows = block_rows;
  sc.emit_bound = 1;
  for (int g = 0; g < n_blocks; ++g) {
    HGR_CHECK_ARG(val_blocks[g] && idx_blocks[g] && bound_blocks[g], "hgr_score_topk_splits_scatter_bounded: null block %d", g);
    sc.val[g] = val_blocks[g];
    sc.idx[g] = idx_blocks[g];
    sc.bound[g] = bound_blocks[g];
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (C == 0) {
    // no rows on this rank: every split stores (-inf, -1) lists and a -inf bound (the merge of zero lists)
    for (int sp = 0; sp < n_splits; ++sp) {
      OutScatter split_sc = sc;
      for (int g = 0; g < n_blocks; ++g) {
        split_sc.val[g] += sp * split_stride;
        split_sc.idx[g] += sp * split_stride;
        split_sc.bound[g] += sp * split_stride;
      }
      rc = merge_zero_lists(B, K, nullptr, nullptr, &split_sc, s);
      if (rc != HGR_OK) return rc;
    }
    return HGR_OK;
  }
  HGR_CHECK_ARG(X && bank, "hgr_score_topk_splits_scatter_bounded: null X / bank");
  HGR_CHECK_ARG(aligned16(X) && aligned16(bank) && aligned16(workspace),
                "hgr_score_topk_splits_scatter_bounded: X/bank/workspace must be 16-byte aligned");
  if (!umma_supported(B, C, D, K))
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_splits_scatter_bounded: shape not supported by the tcgen05 kernel");
  return launch_score_topk_splits_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), col_id,
                                       id_base, nullptr, nullptr, 0, B, C, D, scale, K, gr, group_splits, n_splits,
                                       workspace, workspace_bytes, nullptr, nullptr, nullptr, false, s, &sc,
                                       split_C_total, split_stride);
}

int hgr_score_topk_splits_global_list_len(int64_t B, int64_t C, int64_t D, int K, int n_groups, const int32_t* group_end,
                                          const uint8_t* group_splits, int n_splits, const int64_t* split_C_total) {
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_splits_global_list_len: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  Groups gr;
  int rc = split_table(C, n_groups, group_end, group_splits, n_splits, &gr);
  if (rc != HGR_OK) return rc;
  rc = split_totals(n_splits, split_C_total);
  if (rc != HGR_OK) return rc;
  if (!umma_supported(B, C, D, K))
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_splits_global_list_len: shape not supported by the tcgen05 kernel");
  return umma_split_global_list_len(B, C, D, K, gr, group_splits, n_splits, split_C_total);
}

int hgr_score_topk_plan_shared(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* plan) {
  HGR_CHECK_ARG(plan != nullptr, "hgr_score_topk_plan: null plan");
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_plan: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(grid_share >= 0 && grid_share <= HGR_GRID_SHARE_MAX, "hgr_score_topk_plan: grid share %d outside [0, %d]",
                grid_share, HGR_GRID_SHARE_MAX);
  if (!umma_supported(B, C, D, K)) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_plan: shape not supported by the tcgen05 kernel");
  umma_plan(B, C, D, K, grid_share > 1 ? grid_share : 1, plan);
  return HGR_OK;
}

int hgr_score_topk_plan(int64_t B, int64_t C, int64_t D, int K, int32_t* plan) {
  return hgr_score_topk_plan_shared(B, C, D, K, 1, plan);
}

int hgr_score_topk_grid_share(int64_t B, int64_t C, int64_t D, int K) {
  if (K < 1 || K > HGR_TOPK_MAX || !umma_supported(B, C, D, K)) return 1;
  return umma_grid_share(B, C);
}

int hgr_score_topk_footprint_shared(int64_t B, int64_t C, int64_t D, int K, int grid_share, int x_dtype, int32_t* out) {
  HGR_CHECK_ARG(out != nullptr, "hgr_score_topk_footprint: null out");
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_footprint: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(grid_share >= 0 && grid_share <= HGR_GRID_SHARE_MAX,
                "hgr_score_topk_footprint: grid share %d outside [0, %d]", grid_share, HGR_GRID_SHARE_MAX);
  if (!umma_supported(B, C, D, K)) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_footprint: shape not supported by the tcgen05 kernel");
  const int rc = normalize_rows_footprint(x_dtype, D, out);
  return rc != HGR_OK ? rc : umma_footprint(B, C, D, K, grid_share > 1 ? grid_share : 1, out + 4);
}

int hgr_score_topk_footprint(int64_t B, int64_t C, int64_t D, int K, int x_dtype, int32_t* out) {
  return hgr_score_topk_footprint_shared(B, C, D, K, 1, x_dtype, out);
}

int hgr_score_topk(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, const int32_t* targets,
                   int64_t B, int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                   float* topk_val, int32_t* topk_idx, int64_t* hits, int impl, void* stream) {
  return score_topk_impl(X, bank, col_id, id_base, targets, B, C, D, scale, K, workspace, workspace_bytes, topk_val,
                         topk_idx, hits, impl, stream, nullptr);
}

static int score_topk_scatter_impl(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, int64_t B,
                                   int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                                   int64_t block_rows, int n_blocks, float* const* val_blocks, int32_t* const* idx_blocks,
                                   float* const* bound_blocks, int64_t C_total, int impl, void* stream) {
  HGR_CHECK_ARG(n_blocks >= 1 && n_blocks <= kMaxScatterBlocks, "hgr_score_topk_scatter: n_blocks = %d outside [1, %d]",
                n_blocks, kMaxScatterBlocks);
  HGR_CHECK_ARG(block_rows >= 1 && block_rows * n_blocks >= B, "hgr_score_topk_scatter: %d blocks of %lld rows do not cover B = %lld",
                n_blocks, (long long)block_rows, (long long)B);
  HGR_CHECK_ARG(val_blocks && idx_blocks, "hgr_score_topk_scatter: null block tables");
  // (NO_MERGE with bounds: diagnostics -- the scoring kernel alone with the list length of the global certificate;
  //  nothing is scattered, the block tables are not dereferenced)
  HGR_CHECK_ARG((impl & HGR_IMPL_FLAG_NO_MERGE) == 0 || bound_blocks != nullptr, "hgr_score_topk_scatter: NO_MERGE makes no sense here");
  OutScatter sc;
  sc.n_blocks = n_blocks;
  sc.block_rows = block_rows;
  sc.emit_bound = bound_blocks != nullptr;
  for (int g = 0; g < n_blocks; ++g) {
    HGR_CHECK_ARG(val_blocks[g] && idx_blocks[g], "hgr_score_topk_scatter: null block %d", g);
    HGR_CHECK_ARG(bound_blocks == nullptr || bound_blocks[g], "hgr_score_topk_scatter_bounded: null bound block %d", g);
    sc.val[g] = val_blocks[g];
    sc.idx[g] = idx_blocks[g];
    sc.bound[g] = bound_blocks ? bound_blocks[g] : nullptr;
  }
  return score_topk_impl(X, bank, col_id, id_base, nullptr, B, C, D, scale, K, workspace, workspace_bytes, nullptr, nullptr,
                         nullptr, impl, stream, &sc, C_total);
}

int hgr_score_topk_scatter(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, int64_t B, int64_t C,
                           int64_t D, float scale, int K, void* workspace, size_t workspace_bytes, int64_t block_rows,
                           int n_blocks, float* const* val_blocks, int32_t* const* idx_blocks, int impl, void* stream) {
  return score_topk_scatter_impl(X, bank, col_id, id_base, B, C, D, scale, K, workspace, workspace_bytes, block_rows,
                                 n_blocks, val_blocks, idx_blocks, nullptr, 0, impl, stream);
}

int hgr_score_topk_scatter_bounded(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, int64_t B,
                                   int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                                   int64_t block_rows, int n_blocks, float* const* val_blocks, int32_t* const* idx_blocks,
                                   float* const* bound_blocks, int64_t C_total, int impl, void* stream) {
  HGR_CHECK_ARG(bound_blocks != nullptr, "hgr_score_topk_scatter_bounded: null bound table");
  HGR_CHECK_ARG(C_total >= C, "hgr_score_topk_scatter_bounded: C_total = %lld < C = %lld", (long long)C_total, (long long)C);
  return score_topk_scatter_impl(X, bank, col_id, id_base, B, C, D, scale, K, workspace, workspace_bytes, block_rows,
                                 n_blocks, val_blocks, idx_blocks, bound_blocks, C_total, impl, stream);
}

int hgr_score_topk_global_list_len(int64_t B, int64_t C, int64_t D, int K, int64_t C_total) {
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_score_topk_global_list_len: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  if (!umma_supported(B, C, D, K)) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_global_list_len: shape not supported by the tcgen05 kernel");
  return umma_global_list_len(B, C, D, K, C_total);
}

int hgr_peer_alloc(size_t bytes, void** ptr, unsigned char* handle) {
  HGR_CHECK_ARG(ptr && handle && bytes > 0, "hgr_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == HGR_IPC_HANDLE_BYTES, "IPC handle size");
  void* p = nullptr;
  HGR_CHECK_CUDA(cudaMalloc(&p, bytes));
  HGR_CHECK_CUDA(cudaMemset(p, 0, bytes));
  HGR_CHECK_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return set_error(HGR_ERR_CUDA, "hgr_peer_alloc: cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
  }
  memcpy(handle, &h, sizeof(h));
  *ptr = p;
  return HGR_OK;
}

int hgr_peer_open(const unsigned char* handle, void** ptr) {
  HGR_CHECK_ARG(ptr && handle, "hgr_peer_open: bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  HGR_CHECK_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return HGR_OK;
}

int hgr_peer_close(void* ptr) {
  if (ptr) HGR_CHECK_CUDA(cudaIpcCloseMemHandle(ptr));
  return HGR_OK;
}

int hgr_peer_free(void* ptr) {
  if (ptr) HGR_CHECK_CUDA(cudaFree(ptr));
  return HGR_OK;
}

int hgr_normalize_rows_bcast(const void* E, int e_dtype, int64_t n_rows, int64_t D, int64_t row0, int n_dst,
                             void* const* dst, void* stream) {
  HGR_CHECK_ARG(n_rows >= 0 && row0 >= 0, "hgr_normalize_rows_bcast: negative size");
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_normalize_rows_bcast: D = %lld must be a positive multiple of 8", (long long)D);
  HGR_CHECK_ARG(n_dst >= 1 && n_dst <= kMaxScatterBlocks, "hgr_normalize_rows_bcast: n_dst = %d outside [1, %d]", n_dst,
                kMaxScatterBlocks);
  if (n_rows == 0) return HGR_OK;
  HGR_CHECK_ARG(E && dst, "hgr_normalize_rows_bcast: null pointer");
  for (int g = 0; g < n_dst; ++g)
    HGR_CHECK_ARG(dst[g] && aligned16(dst[g]), "hgr_normalize_rows_bcast: destination %d null or not 16-byte aligned", g);
  HGR_CHECK_ARG(aligned16(E), "hgr_normalize_rows_bcast: E must be 16-byte aligned");
  return launch_normalize_bcast(E, e_dtype, n_rows, D, row0, n_dst, dst, static_cast<cudaStream_t>(stream));
}

int hgr_peer_signal(uint32_t* const* flags, int n, uint32_t* seq, void* stream) {
  HGR_CHECK_ARG(flags && seq, "hgr_peer_signal: null pointer");
  return launch_peer_signal(flags, n, seq, static_cast<cudaStream_t>(stream));
}

int hgr_peer_wait(const uint32_t* flags, int n, uint32_t* seq, void* stream) {
  HGR_CHECK_ARG(flags && seq, "hgr_peer_wait: null pointer");
  return launch_peer_wait(flags, n, seq, static_cast<cudaStream_t>(stream));
}

// P lists of K entries per row (node ids), merged and counted: hgr_topk_merge, and hgr_topk_merge_certified before it
// adds its certificate.
static MergeArgs list_merge_args(const float* part_val, const int32_t* part_idx, int64_t P, int64_t B, int K,
                                 int64_t part_stride, const int32_t* targets, float* topk_val, int32_t* topk_idx,
                                 int64_t* hits) {
  MergeArgs m{};
  m.part_val = part_val;
  m.part_idx = part_idx;
  m.P = P;
  m.B = B;
  m.KL = K;
  m.K = K;
  m.part_stride = part_stride;
  m.scale = 1.f;
  m.targets = targets;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  m.hits = hits;
  return m;
}

int hgr_topk_merge(const float* part_val, const int32_t* part_idx, int64_t P, int64_t B, int K, int64_t part_stride,
                   const int32_t* targets, float* topk_val, int32_t* topk_idx, int64_t* hits, void* stream) {
  HGR_CHECK_ARG(P >= 0 && B >= 0, "hgr_topk_merge: negative size");
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_topk_merge: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(topk_val && topk_idx, "hgr_topk_merge: null output");
  HGR_CHECK_ARG(P == 0 || (part_val && part_idx), "hgr_topk_merge: null parts");
  HGR_CHECK_ARG(part_stride == 0 || part_stride >= B * K, "hgr_topk_merge: part_stride < B*K");
  return launch_topk_merge(list_merge_args(part_val, part_idx, P, B, K, part_stride, targets, topk_val, topk_idx, hits),
                           static_cast<cudaStream_t>(stream));
}

int hgr_topk_merge_certified(const float* part_val, const int32_t* part_idx, const float* part_bound, int64_t P, int64_t B,
                             int K, int64_t part_stride, int64_t bound_stride, const int32_t* targets, float* topk_val,
                             int32_t* topk_idx, int64_t* hits, const void* X, int64_t D, const hgr_shard_t* shards,
                             float scale, unsigned int* repair_count, void* stream) {
  HGR_CHECK_ARG(P >= 1 && P <= kMaxScatterBlocks && B >= 0, "hgr_topk_merge_certified: P = %lld outside [1, %d]", (long long)P,
                kMaxScatterBlocks);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_topk_merge_certified: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(topk_val && topk_idx && part_val && part_idx && part_bound, "hgr_topk_merge_certified: null lists / bounds / output");
  HGR_CHECK_ARG(X && shards && D > 0 && D % 8 == 0 && aligned16(X), "hgr_topk_merge_certified: the repair needs X (16-byte aligned, D %% 8 == 0) and the shard table");
  HGR_CHECK_ARG(part_stride == 0 || part_stride >= B * K, "hgr_topk_merge_certified: part_stride < B*K");
  HGR_CHECK_ARG(bound_stride >= B, "hgr_topk_merge_certified: bound_stride < B");
  HGR_CHECK_ARG(scale > 0.f, "hgr_topk_merge_certified: scale must be > 0");
  MergeArgs m = list_merge_args(part_val, part_idx, P, B, K, part_stride, targets, topk_val, topk_idx, hits);
  m.part_bound = part_bound;
  m.bound_stride = bound_stride;
  m.shards = shards;
  m.xrows = X;
  m.xD8 = static_cast<int>(D / 8);
  m.shard_scale = scale;
  m.repair_count = repair_count;
  return launch_topk_merge(m, static_cast<cudaStream_t>(stream));
}

int hgr_topk_merge_splits_certified(const float* part_val, const int32_t* part_idx, const float* part_bound, int64_t P,
                                    int64_t B, int K, int n_splits, int64_t part_stride, int64_t bound_stride,
                                    int64_t split_stride, const int32_t* targets, const uint8_t* node_splits,
                                    int64_t n_nodes, float* topk_val, int32_t* topk_idx, int64_t* counts, const void* X,
                                    int64_t D, const hgr_shard_t* shards, float scale, unsigned int* repair_count,
                                    void* stream) {
  HGR_CHECK_ARG(P >= 1 && P <= kMaxScatterBlocks && B >= 0, "hgr_topk_merge_splits_certified: P = %lld outside [1, %d]",
                (long long)P, kMaxScatterBlocks);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_topk_merge_splits_certified: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(n_splits >= 1 && n_splits <= kMaxSplits, "hgr_topk_merge_splits_certified: %d splits outside [1, %d]",
                n_splits, kMaxSplits);
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(topk_val && topk_idx && part_val && part_idx && part_bound,
                "hgr_topk_merge_splits_certified: null lists / bounds / output");
  HGR_CHECK_ARG(node_splits && n_nodes > 0, "hgr_topk_merge_splits_certified: the repair needs node_splits");
  HGR_CHECK_ARG(counts == nullptr || targets, "hgr_topk_merge_splits_certified: counting needs targets");
  HGR_CHECK_ARG(X && shards && D > 0 && D % 8 == 0 && aligned16(X),
                "hgr_topk_merge_splits_certified: the repair needs X (16-byte aligned, D %% 8 == 0) and the shard table");
  HGR_CHECK_ARG(part_stride >= B * K, "hgr_topk_merge_splits_certified: part_stride < B*K");
  HGR_CHECK_ARG(bound_stride >= B, "hgr_topk_merge_splits_certified: bound_stride < B");
  // value lists, id lists and bounds of a split all sit at + s * split_stride: its area spans all three
  HGR_CHECK_ARG(n_splits == 1 || split_stride >= 2 * P * part_stride + P * bound_stride,
                "hgr_topk_merge_splits_certified: split_stride %lld < %lld: the areas of two splits overlap",
                (long long)split_stride, (long long)(2 * P * part_stride + P * bound_stride));
  HGR_CHECK_ARG(scale > 0.f, "hgr_topk_merge_splits_certified: scale must be > 0");
  SplitCertArgs m{};
  m.part_val = part_val;
  m.part_idx = part_idx;
  m.part_bound = part_bound;
  m.P = P;
  m.B = B;
  m.K = K;
  m.S = n_splits;
  m.part_stride = part_stride;
  m.bound_stride = bound_stride;
  m.split_stride = split_stride;
  m.targets = targets;
  m.node_splits = node_splits;
  m.n_nodes = n_nodes;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  m.counts = counts;
  m.shards = shards;
  m.xrows = X;
  m.xD8 = static_cast<int>(D / 8);
  m.scale = scale;
  m.repair_count = repair_count;
  return launch_topk_split_merge_certified(m, static_cast<cudaStream_t>(stream));
}

int64_t hgr_sample_replay(const uint32_t* words, int64_t n_words, int64_t n, int64_t k, int64_t setsize, int32_t* out_pos,
                          int32_t* scratch) {
  if (!words || !out_pos || !scratch || n < 0 || k < 0 || k > n || n >= (int64_t(1) << 31)) return -2;
  auto bit_length = [](uint32_t v) { return v == 0 ? 0 : 32 - __builtin_clz(v); };
  int64_t p = 0;
  if (n <= setsize) {
    for (int64_t i = 0; i < n; ++i) scratch[i] = static_cast<int32_t>(i);
    for (int64_t i = 0; i < k; ++i) {
      const uint32_t left = static_cast<uint32_t>(n - i);
      const int sh = 32 - bit_length(left);
      uint32_t r;
      do {
        if (p >= n_words) return -1;
        r = words[p++] >> sh;
      } while (r >= left);
      out_pos[i] = scratch[r];
      scratch[r] = scratch[left - 1];
    }
    return p;
  }
  for (int64_t i = 0; i < n; ++i) scratch[i] = 0;
  const int sh = 32 - bit_length(static_cast<uint32_t>(n));
  for (int64_t i = 0; i < k; ++i) {
    uint32_t r;
    do {
      do {
        if (p >= n_words) return -1;
        r = words[p++] >> sh;
      } while (r >= static_cast<uint32_t>(n));
    } while (scratch[r]);
    scratch[r] = 1;
    out_pos[i] = static_cast<int32_t>(r);
  }
  return p;
}

int64_t hgr_sample_replay_many(const uint32_t* words, int64_t n_words, int64_t count, const int64_t* n, const int64_t* k,
                               int32_t* out_pos, int32_t* scratch) {
  if (!n || !k || count < 0) return -2;
  int64_t used = 0, off = 0;
  for (int64_t c = 0; c < count; ++c) {
    int64_t setsize = 21;                       // CPython: 21, + 4 ** ceil(log(3 k, 4)) when k > 5
    if (k[c] > 5) {
      int64_t p4 = 1;
      while (p4 < 3 * k[c]) p4 *= 4;
      setsize += p4;
    }
    const int64_t r = hgr_sample_replay(words + used, n_words - used, n[c], k[c], setsize, out_pos + off, scratch);
    if (r < 0) return r;
    used += r;
    off += k[c];
  }
  return used;
}

int64_t hgr_om_plan(const uint32_t* words, int64_t n_words, int64_t T, const int64_t* const* cand, const int64_t* n_cand,
                    const int64_t* anchor, int64_t num_compare, int64_t n_nodes, int32_t* set_ptr, int32_t* set_col,
                    int32_t* label_pos, int32_t* union_ids, int64_t* counts, int32_t* scratch) {
  if (!cand || !n_cand || !anchor || !set_ptr || !set_col || !label_pos || !union_ids || !counts || !scratch || T < 0 ||
      num_compare < 0 || n_nodes <= 0 || n_nodes >= (int64_t(1) << 31))
    return -2;
  int64_t max_n = 0;
  for (int64_t t = 0; t < T; ++t) {
    if (n_cand[t] < 0 || (n_cand[t] > 0 && !cand[t]) || anchor[t] < 0 || anchor[t] >= n_nodes) return -2;
    max_n = n_cand[t] > max_n ? n_cand[t] : max_n;
  }
  int32_t* mark = scratch;                 // [n_nodes]: 0, then union position + 1
  int32_t* pool = scratch + n_nodes;       // [max_n]
  int32_t* pos = pool + max_n;             // [num_compare]
  for (int64_t i = 0; i < n_nodes; ++i) mark[i] = 0;
  int64_t setsize = 21;                    // CPython: 21, + 4 ** ceil(log(3 k, 4)) when k > 5
  if (num_compare > 5) {
    int64_t p4 = 1;
    while (p4 < 3 * num_compare) p4 *= 4;
    setsize += p4;
  }
  int64_t used = 0;
  set_ptr[0] = 0;
  for (int64_t t = 0; t < T; ++t) {
    int32_t* out = set_col + set_ptr[t];
    int64_t m = 0;
    if (n_cand[t] > num_compare) {
      if (words == nullptr) return -2;
      const int64_t r = hgr_sample_replay(words + used, n_words - used, n_cand[t], num_compare, setsize, pos, pool);
      if (r < 0) return r;
      used += r;
      for (int64_t i = 0; i < num_compare; ++i) out[i] = static_cast<int32_t>(cand[t][pos[i]]);
      m = num_compare;
    } else {
      for (int64_t i = 0; i < n_cand[t]; ++i) out[i] = static_cast<int32_t>(cand[t][i]);
      m = n_cand[t];
    }
    int64_t lp = -1;
    for (int64_t i = 0; i < m && lp < 0; ++i)
      if (out[i] == anchor[t]) lp = i;
    if (lp < 0) {
      out[m] = static_cast<int32_t>(anchor[t]);
      lp = m++;
    }
    label_pos[t] = static_cast<int32_t>(lp);
    for (int64_t i = 0; i < m; ++i) {
      if (out[i] < 0 || out[i] >= n_nodes) return -2;
      mark[out[i]] = 1;
    }
    set_ptr[t + 1] = set_ptr[t] + static_cast<int32_t>(m);
  }
  int64_t nu = 0;
  for (int64_t i = 0; i < n_nodes; ++i)
    if (mark[i]) {
      union_ids[nu] = static_cast<int32_t>(i);
      mark[i] = static_cast<int32_t>(++nu);
    }
  const int64_t n_col = set_ptr[T];
  for (int64_t e = 0; e < n_col; ++e) set_col[e] = mark[set_col[e]] - 1;
  counts[0] = n_col;
  counts[1] = nu;
  return used;
}

int hgr_logits_dense(const void* X, const void* bank, int64_t B, int64_t C, int64_t D, float scale, float* out,
                     int64_t ldo, int impl, void* stream) {
  HGR_CHECK_ARG(B >= 0 && C >= 0, "hgr_logits_dense: negative size");
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_logits_dense: D = %lld must be a positive multiple of 8", (long long)D);
  if (B == 0 || C == 0) return HGR_OK;
  HGR_CHECK_ARG(X && bank && out, "hgr_logits_dense: null pointer");
  HGR_CHECK_ARG(ldo >= C, "hgr_logits_dense: ldo < C");
  HGR_CHECK_ARG(aligned16(X) && aligned16(bank), "hgr_logits_dense: X/bank must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int which = pick_impl(impl, B, C, D, 1);
  if (which == HGR_IMPL_TCGEN05)
    return launch_logits_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), B, C, D,
                              scale, out, ldo, s);
  if (which == HGR_IMPL_SIMT)
    return launch_logits_simt(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank), B, C, D,
                              scale, out, ldo, s);
  return set_error(HGR_ERR_BAD_ARG, "hgr_logits_dense: unknown impl %d", impl);
}

int hgr_hier_metrics_fused_rows(const void* X, const void* bank_sorted, int64_t B, int64_t M, int64_t D,
                                const int32_t* level_end, int n_levels, const int32_t* sorted_to_pos,
                                const int32_t* first_out, const int32_t* targets, int64_t n_nodes,
                                const int32_t* chain_ptr, const int32_t* chain_pos, const int32_t* chain_level,
                                const uint8_t* node_splits, int n_sets, void* workspace, size_t workspace_bytes,
                                int32_t* lvl_idx, int32_t* top1, int64_t* counts, void* stream) {
  HGR_CHECK_ARG(B >= 0 && M > 0 && M <= (int64_t(1) << 31) - 512, "hgr_hier_metrics_fused_rows: bad sizes B=%lld M=%lld",
                (long long)B, (long long)M);
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_hier_metrics_fused_rows: D = %lld must be a positive multiple of 8", (long long)D);
  HGR_CHECK_ARG(n_nodes > 0 && n_nodes < (int64_t(1) << 31) - 1, "hgr_hier_metrics_fused_rows: n_nodes = %lld",
                (long long)n_nodes);
  HGR_CHECK_ARG(n_levels >= 1 && n_levels <= 32, "hgr_hier_metrics_fused_rows: %d levels outside [1, 32]", n_levels);
  HGR_CHECK_ARG(n_sets >= 1 && n_sets <= (node_splits ? kMaxSplits : 1),
                "hgr_hier_metrics_fused_rows: %d counter sets outside [1, %d] (%s node_splits)", n_sets,
                node_splits ? kMaxSplits : 1, node_splits ? "with" : "without");
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(X && bank_sorted && level_end && sorted_to_pos && first_out && targets && chain_ptr && chain_pos &&
                    chain_level && counts && workspace,
                "hgr_hier_metrics_fused_rows: null pointer");
  HGR_CHECK_ARG(aligned16(X) && aligned16(bank_sorted) && aligned16(workspace),
                "hgr_hier_metrics_fused_rows: X / bank / workspace must be 16-byte aligned");
  HGR_CHECK_ARG(workspace_bytes >= static_cast<size_t>(B) * n_levels * 8, "hgr_hier_metrics_fused_rows: workspace %zu < %zu bytes",
                workspace_bytes, static_cast<size_t>(B) * n_levels * 8);
  if (!umma_supported(B, M, D, 1))
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics_fused_rows: shape not supported by the tcgen05 kernel");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned long long* best = static_cast<unsigned long long*>(workspace);
  const int rc = launch_level_argmax_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank_sorted), B, M,
                                          D, level_end, n_levels, best, s);
  if (rc != HGR_OK) return rc;
  return launch_hier_finish_rows(best, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr, chain_pos,
                                 chain_level, node_splits, n_sets, lvl_idx, top1, counts, s);
}

int hgr_hier_level_scatter(const void* X, const void* bank_shard, int64_t B, int64_t M_r, int64_t D,
                           const int32_t* level_end_local, int n_levels, int64_t row_base, void* workspace,
                           size_t workspace_bytes, int64_t block_rows, int n_blocks, uint64_t* const* dst_blocks,
                           void* stream) {
  HGR_CHECK_ARG(B >= 0 && M_r >= 0 && M_r < (int64_t(1) << 31) - 512, "hgr_hier_level_scatter: bad sizes B=%lld M_r=%lld",
                (long long)B, (long long)M_r);
  HGR_CHECK_ARG(D > 0 && D % 8 == 0, "hgr_hier_level_scatter: D = %lld must be a positive multiple of 8", (long long)D);
  HGR_CHECK_ARG(n_levels >= 1 && n_levels <= 32, "hgr_hier_level_scatter: %d levels outside [1, 32]", n_levels);
  HGR_CHECK_ARG(row_base >= 0 && row_base + M_r < (int64_t(1) << 31) - 512,
                "hgr_hier_level_scatter: row_base = %lld puts the shard outside the global sorted bank", (long long)row_base);
  HGR_CHECK_ARG(n_blocks >= 1 && n_blocks <= kMaxScatterBlocks, "hgr_hier_level_scatter: n_blocks = %d outside [1, %d]",
                n_blocks, kMaxScatterBlocks);
  HGR_CHECK_ARG(block_rows >= 1 && block_rows * n_blocks >= B, "hgr_hier_level_scatter: %d blocks of %lld rows do not cover B = %lld",
                n_blocks, (long long)block_rows, (long long)B);
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(dst_blocks && workspace && (M_r == 0 || (X && bank_shard && level_end_local)),
                "hgr_hier_level_scatter: null pointer");
  for (int g = 0; g < n_blocks; ++g)
    HGR_CHECK_ARG(dst_blocks[g] && (reinterpret_cast<uintptr_t>(dst_blocks[g]) & 7u) == 0,
                  "hgr_hier_level_scatter: destination %d null or not 8-byte aligned", g);
  HGR_CHECK_ARG(aligned16(workspace) && (M_r == 0 || (aligned16(X) && aligned16(bank_shard))),
                "hgr_hier_level_scatter: X / bank / workspace must be 16-byte aligned");
  HGR_CHECK_ARG(workspace_bytes >= static_cast<size_t>(B) * n_levels * 8, "hgr_hier_level_scatter: workspace %zu < %zu bytes",
                workspace_bytes, static_cast<size_t>(B) * n_levels * 8);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned long long* best = static_cast<unsigned long long*>(workspace);
  if (M_r > 0) {          // an empty shard has no GEMM: its workspace is still all zero and the push stores zeros
    if (!umma_supported(B, M_r, D, 1))
      return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_level_scatter: shape not supported by the tcgen05 kernel");
    const int rc = launch_level_argmax_umma(static_cast<const __nv_bfloat16*>(X), static_cast<const __nv_bfloat16*>(bank_shard),
                                            B, M_r, D, level_end_local, n_levels, best, s);
    if (rc != HGR_OK) return rc;
  }
  return launch_hier_push(best, B, n_levels, row_base, block_rows, n_blocks,
                          reinterpret_cast<unsigned long long* const*>(dst_blocks), s);
}

int hgr_hier_finish_rows_gathered(const uint64_t* parts, int n_parts, int64_t part_stride, int64_t n_rows, int64_t M,
                                  int n_levels, const int32_t* sorted_to_pos, const int32_t* first_out,
                                  const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                                  const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits,
                                  int n_sets, int32_t* lvl_idx, int32_t* top1, int64_t* counts, void* stream) {
  HGR_CHECK_ARG(n_rows >= 0 && M > 0 && M <= (int64_t(1) << 31) - 512, "hgr_hier_finish_rows_gathered: bad sizes n_rows=%lld M=%lld",
                (long long)n_rows, (long long)M);
  HGR_CHECK_ARG(n_nodes > 0 && n_nodes < (int64_t(1) << 31) - 1, "hgr_hier_finish_rows_gathered: n_nodes = %lld",
                (long long)n_nodes);
  HGR_CHECK_ARG(n_levels >= 1 && n_levels <= 32, "hgr_hier_finish_rows_gathered: %d levels outside [1, 32]", n_levels);
  HGR_CHECK_ARG(n_parts >= 1 && n_parts <= kMaxScatterBlocks, "hgr_hier_finish_rows_gathered: n_parts = %d outside [1, %d]",
                n_parts, kMaxScatterBlocks);
  HGR_CHECK_ARG(n_sets >= 1 && n_sets <= (node_splits ? kMaxSplits : 1),
                "hgr_hier_finish_rows_gathered: %d counter sets outside [1, %d] (%s node_splits)", n_sets,
                node_splits ? kMaxSplits : 1, node_splits ? "with" : "without");
  HGR_CHECK_ARG(part_stride >= n_rows * n_levels, "hgr_hier_finish_rows_gathered: part_stride < n_rows * n_levels");
  if (n_rows == 0) return HGR_OK;
  HGR_CHECK_ARG(parts && sorted_to_pos && first_out && targets && chain_ptr && chain_pos && chain_level && counts,
                "hgr_hier_finish_rows_gathered: null pointer");
  HGR_CHECK_ARG((reinterpret_cast<uintptr_t>(parts) & 7u) == 0, "hgr_hier_finish_rows_gathered: parts must be 8-byte aligned");
  return launch_hier_finish_gathered(reinterpret_cast<const unsigned long long*>(parts), n_parts, part_stride, n_rows, M,
                                     n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr, chain_pos, chain_level,
                                     node_splits, n_sets, lvl_idx, top1, counts, static_cast<cudaStream_t>(stream));
}

// main.py:135-148 extended from "label in the first k" to the hierarchy distance of the first k (hier_mistakes.cu).
int hgr_hier_mistakes(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                      const uint8_t* node_splits, const int32_t* chain_ptr, const int32_t* chain_node, int64_t n_nodes,
                      int64_t* counts, void* stream) {
  HGR_CHECK_ARG(B >= 0 && B <= (int64_t(1) << 31) - 1, "hgr_hier_mistakes: bad size B=%lld", (long long)B);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_hier_mistakes: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(n_nodes > 0 && n_nodes < (int64_t(1) << 31) - 1, "hgr_hier_mistakes: n_nodes = %lld", (long long)n_nodes);
  HGR_CHECK_ARG(n_sets >= 1 && n_sets <= (node_splits ? kMaxSplits : 1),
                "hgr_hier_mistakes: %d list sets outside [1, %d] (%s node_splits)", n_sets, node_splits ? kMaxSplits : 1,
                node_splits ? "with" : "without");
  HGR_CHECK_ARG(n_sets == 1 || set_stride >= B * K, "hgr_hier_mistakes: set_stride %lld < B * K = %lld",
                (long long)set_stride, (long long)(B * K));
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(topk_idx && targets && chain_ptr && chain_node && counts, "hgr_hier_mistakes: null pointer");
  HGR_CHECK_ARG((reinterpret_cast<uintptr_t>(counts) & 7u) == 0, "hgr_hier_mistakes: counts must be 8-byte aligned");
  return launch_hier_mistakes(topk_idx, B, K, set_stride, n_sets, targets, node_splits, chain_ptr, chain_node, n_nodes,
                              counts, static_cast<cudaStream_t>(stream));
}

// main.py:135-148 counted per label: the table behind class-averaged Hit@k (class_hits.cu).
int hgr_class_hits(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                   const uint8_t* node_splits, int64_t n_nodes, int64_t* counts, void* stream) {
  HGR_CHECK_ARG(B >= 0 && B <= (int64_t(1) << 31) - 1, "hgr_class_hits: bad size B=%lld", (long long)B);
  HGR_CHECK_ARG(K >= 1 && K <= HGR_TOPK_MAX, "hgr_class_hits: K = %d outside [1, %d]", K, HGR_TOPK_MAX);
  HGR_CHECK_ARG(n_nodes > 0 && n_nodes < (int64_t(1) << 31) - 1, "hgr_class_hits: n_nodes = %lld", (long long)n_nodes);
  HGR_CHECK_ARG(n_sets >= 1 && n_sets <= (node_splits ? kMaxSplits : 1),
                "hgr_class_hits: %d list sets outside [1, %d] (%s node_splits)", n_sets, node_splits ? kMaxSplits : 1,
                node_splits ? "with" : "without");
  HGR_CHECK_ARG(n_sets == 1 || set_stride >= B * K, "hgr_class_hits: set_stride %lld < B * K = %lld",
                (long long)set_stride, (long long)(B * K));
  if (B == 0) return HGR_OK;
  HGR_CHECK_ARG(topk_idx && targets && counts, "hgr_class_hits: null pointer");
  HGR_CHECK_ARG((reinterpret_cast<uintptr_t>(counts) & 7u) == 0, "hgr_class_hits: counts must be 8-byte aligned");
  return launch_class_hits(topk_idx, B, K, set_stride, n_sets, targets, node_splits, n_nodes, counts,
                           static_cast<cudaStream_t>(stream));
}

size_t hgr_masked_ce_workspace_bytes(int64_t B, int64_t U, int64_t T) { return masked_ce_workspace_bytes(B, U, T) + 16; }

int hgr_masked_ce(const float* logits, int64_t ldl, int64_t B, int64_t U, const int32_t* set_ptr, const int32_t* set_col,
                  const int32_t* label_pos, const float* weight, int64_t T, float* loss, float* dlogits, void* workspace,
                  size_t workspace_bytes, void* stream) {
  HGR_CHECK_ARG(B > 0 && U > 0 && T >= 0, "hgr_masked_ce: bad sizes B=%lld U=%lld T=%lld", (long long)B, (long long)U, (long long)T);
  HGR_CHECK_ARG(ldl >= U, "hgr_masked_ce: ldl < U");
  if (T == 0) {
    // no set: the loss is empty and the gradient is zero everywhere, still overwritten as documented
    if (dlogits)
      HGR_CHECK_CUDA(cudaMemset2DAsync(dlogits, static_cast<size_t>(ldl) * sizeof(float), 0,
                                       static_cast<size_t>(U) * sizeof(float), static_cast<size_t>(B),
                                       static_cast<cudaStream_t>(stream)));
    return HGR_OK;
  }
  HGR_CHECK_ARG(logits && set_ptr && set_col && label_pos && weight && loss, "hgr_masked_ce: null pointer");
  return launch_masked_ce(logits, ldl, B, U, set_ptr, set_col, label_pos, weight, T, loss, dlogits, workspace,
                          workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t hgr_om_backward_workspace_bytes(int64_t B, int64_t U, int64_t D) { return om_backward_workspace_bytes(B, U, D) + 16; }

int hgr_om_backward(const float* dlogits, const float* logits, int64_t ldl, int64_t B, int64_t U, int64_t D, const void* x,
                    const float* x_norm, const void* tn, const float* t_norm, float scale, float* d_img, float* d_text,
                    float* d_log_scale, void* workspace, size_t workspace_bytes, void* stream) {
  HGR_CHECK_ARG(B > 0 && U > 0 && D > 0, "hgr_om_backward: bad sizes B=%lld U=%lld D=%lld", (long long)B, (long long)U, (long long)D);
  HGR_CHECK_ARG(ldl >= U, "hgr_om_backward: ldl < U");
  HGR_CHECK_ARG(dlogits && logits && x && x_norm && tn && t_norm && d_img && d_text, "hgr_om_backward: null pointer");
  HGR_CHECK_ARG(aligned16(x) && aligned16(tn) && aligned16(d_img) && aligned16(d_text) && aligned16(workspace),
                "hgr_om_backward: x / tn / d_img / d_text / workspace must be 16-byte aligned");
  return launch_om_backward(dlogits, logits, ldl, B, U, D, static_cast<const __nv_bfloat16*>(x), x_norm,
                            static_cast<const __nv_bfloat16*>(tn), t_norm, scale, d_img, d_text, d_log_scale, workspace,
                            workspace_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
