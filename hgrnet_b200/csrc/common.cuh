// Shared host-side plumbing of libhgr_b200: error reporting, launch accounting, constants.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "../../include/hgr_b200.h"
#include "sched.cuh"

namespace hgr {

constexpr int kNumSMsB200 = 148;
// Hit@k cut-offs of the eval loop, main.py:120
__host__ __device__ constexpr int hit_cut(int c) { return c == 0 ? 1 : c == 1 ? 2 : c == 2 ? 5 : c == 3 ? 10 : 20; }

int set_error(int code, const char* fmt, ...);
void count_launch(int n = 1);
int num_sms();  // SM count of the current device (cached)

#define HGR_CHECK_ARG(cond, ...)                                   \
  do {                                                             \
    if (!(cond)) return ::hgr::set_error(HGR_ERR_BAD_ARG, __VA_ARGS__); \
  } while (0)

#define HGR_CHECK_CUDA(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess)                                                              \
      return ::hgr::set_error(HGR_ERR_CUDA, "%s failed: %s (%d) at %s:%d", #expr,       \
                              cudaGetErrorString(_e), (int)_e, __FILE__, __LINE__);     \
  } while (0)

#define HGR_CHECK_LAUNCH()                                                              \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess)                                                              \
      return ::hgr::set_error(HGR_ERR_CUDA, "kernel launch failed: %s (%d) at %s:%d",   \
                              cudaGetErrorString(_e), (int)_e, __FILE__, __LINE__);     \
    ::hgr::count_launch();                                                              \
  } while (0)

// Total order used everywhere a top-k list is kept: larger value first; among equal values
// the smaller tag (bank row / part position) first.  NaNs never enter a list (v > x is false).
struct Cand {
  float v;
  int32_t i;
};

// ---- entry points implemented in the individual .cu files (called from hgr_abi.cu) ----
int launch_aggregate_normalize(const void* E, int e_dtype, int64_t n_src, int64_t D,
                               const int32_t* rowptr, const int32_t* col, const float* w,
                               const int32_t* row_map, int64_t n_out, void* out, int out_dtype,
                               float* out_norm, cudaStream_t stream);

// Arguments of the list-merge kernel (topk_merge.cu).
//  * public use (hgr_topk_merge / SIMT path): `P` lists of length KL == K per row, all valid.
//  * tcgen05 path: `use_sched` -- row tile mt owns sched.parts(mt) lists of length KL (the partial lists of
//    each worker segment).  When KL < K the lists are SPECULATIVE (narrower than K); the merge
//    certifies every row (a full list whose last entry still beats the merged K-th value may hide candidates)
//    and re-scans uncertified rows exactly on the CUDA cores, for which it needs X / bank.
// Row-block scatter of the final lists: rows [g * block_rows, (g + 1) * block_rows) go to val[g] / idx[g] (each a
// dense [block_rows, K] array).  The pointers may be PEER memory (another GPU's exchange buffer mapped over NVLink):
// the class-sharded head writes every rank's candidates straight into the buffers of the rank that owns the rows.
constexpr int kMaxScatterBlocks = 16;
// `bound` (global certificate of the class-sharded head, see hgr_score_topk_scatter_bounded): next to the final list of
// a row the producer stores an upper bound of every candidate its narrow lists may have dropped (-inf: none).
struct OutScatter {
  int n_blocks = 0;
  int emit_bound = 0;
  int64_t block_rows = 0;
  float* val[kMaxScatterBlocks];
  int32_t* idx[kMaxScatterBlocks];
  float* bound[kMaxScatterBlocks];
};

struct MergeArgs {
  const float* part_val;
  const int32_t* part_idx;
  int64_t P, B;
  int KL, K;
  int64_t part_stride;      // elements between consecutive lists (0 -> B * KL)
  int use_sched;
  Sched sched;
  const int32_t* col_id;
  int32_t id_base;
  float scale;
  const int32_t* targets;
  float* topk_val;
  int32_t* topk_idx;
  int64_t* hits;
  const void* X;            // [B, D] bf16 -- exact re-scan only
  const void* bank;         // [C, D] bf16
  int64_t C;
  int D8;
  unsigned int* rescan_count;  // optional statistics: number of rows re-scanned
  OutScatter scatter;          // n_blocks > 0: replaces topk_val / topk_idx
  // candidate lists of the floor-sketch epilogue (sketch_epi.cuh): list p of a row holds sk_cnt[p * B + row] <= sk_cap
  // unsorted (value bits, bank row) entries at sk_part[(p * B + row) * sk_cap]; replaces part_val / part_idx / KL
  const uint2* sk_part = nullptr;
  const int32_t* sk_cnt = nullptr;
  int sk_cap = 0;
  // owner side of the global certificate (hgr_topk_merge_certified): list p comes from class shard p, and everything
  // that shard dropped for a row is <= part_bound[p * bound_stride + row].  A row whose merged K-th value does not
  // beat every bound strictly is repaired exactly: the doubtful shards are re-scanned (shards[p], device memory,
  // possibly a peer's bank over NVLink) with the row's features xrows[row] and the producers' logit scale.
  const float* part_bound = nullptr;
  int64_t bound_stride = 0;
  const hgr_shard_t* shards = nullptr;
  const void* xrows = nullptr;
  int xD8 = 0;
  float shard_scale = 1.f;
  unsigned int* repair_count = nullptr;
};
int launch_topk_merge(const MergeArgs& args, cudaStream_t stream);
// {threads, registers per thread, static shared memory, dynamic shared memory} of the merge launch_topk_merge runs on
// the scoring kernel's own P lists of KL entries per row (register merges only)
int merge_kernel_footprint(int64_t P, int KL, int32_t* out);

// Arguments of the per-split merge (hgr_score_topk_splits, topk_merge.cu): the scoring kernel's lists on the grouped
// schedule, group_parts(mt) lists of length KL per row, list slot p of row tile mt covering the bank rows
// group_slot_range(p) of one group.  Split s is the union of the groups g with bit s of group_splits[g].
constexpr int kMaxSplits = 8;
struct SplitMergeArgs {
  const float* part_val;       // [slots][B][KL]
  const int32_t* part_idx;     // [slots][B][KL] bank rows
  int64_t B, C;
  int KL, K, S;
  Sched sched;
  Groups groups;
  uint8_t group_splits[kMaxGroups];
  const int32_t* col_id;
  int32_t id_base;
  float scale;
  const int32_t* targets;      // [B] node ids, or null
  const uint8_t* node_splits;  // [n_nodes] split bits of every node
  int64_t n_nodes;
  float* topk_val;             // [S][B][K]
  int32_t* topk_idx;           // [S][B][K] node ids
  int64_t* counts;             // [S][HGR_NUM_HITS + 1]: Hit@{1,2,5,10,20}, rows; or null
  const void* X;               // [B, D] bf16 -- exact re-scan only
  const void* bank;            // [C, D] bf16
  int D8;
  unsigned int* rescan_count;  // (row, split) pairs re-scanned
  // bounded scatter (hgr_score_topk_splits_scatter_bounded): instead of topk_val / topk_idx / counts, split s of row
  // block g goes to scatter.val[g] / idx[g] / bound[g] + s * split_stride elements; no local certificate, no repair
  OutScatter scatter;
  int64_t split_stride;
};
int launch_topk_split_merge(const SplitMergeArgs& args, cudaStream_t stream);

// Owner side of the class-sharded per-split certificate (hgr_topk_merge_splits_certified): split s of list p (class
// shard p) sits at part_val / part_idx + s * split_stride + p * part_stride + row * K (node ids, scaled values), its
// bound at part_bound + s * split_stride + p * bound_stride + row.
struct SplitCertArgs {
  const float* part_val;
  const int32_t* part_idx;
  const float* part_bound;
  int64_t P, B;
  int K, S;
  int64_t part_stride, bound_stride, split_stride;
  const int32_t* targets;      // [B] node ids, or null
  const uint8_t* node_splits;  // [n_nodes] split bits of every node
  int64_t n_nodes;
  float* topk_val;             // [S][B][K]
  int32_t* topk_idx;           // [S][B][K] node ids
  int64_t* counts;             // [S][HGR_NUM_HITS + 1], or null
  const hgr_shard_t* shards;   // [P] the shards' banks (peer memory) for the exact repair
  const void* xrows;           // [B, D] bf16
  int xD8;
  float scale;
  unsigned int* repair_count;  // (row, split) pairs repaired
};
int launch_topk_split_merge_certified(const SplitCertArgs& args, cudaStream_t stream);

// Bytes at the front of the per-stream scoring workspace that carry state from one tcgen05 scoring call to the next
// (umma_common.cuh: statistics, the floor-sketch epoch, timeline stamps); every other user of the workspace starts
// behind them.
constexpr int kScoreWsHeaderBytes = 64 + 256 * 32 * 8;
size_t simt_score_workspace_bytes(int64_t B, int64_t C, int K);
int launch_score_topk_simt(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                           int32_t id_base, const int32_t* targets, int64_t B, int64_t C, int64_t D,
                           float scale, int K, void* ws, size_t ws_bytes, float* topk_val,
                           int32_t* topk_idx, int64_t* hits, cudaStream_t stream,
                           const OutScatter* scatter = nullptr);
int launch_logits_simt(const __nv_bfloat16* X, const __nv_bfloat16* bank, int64_t B, int64_t C,
                       int64_t D, float scale, float* out, int64_t ldo, cudaStream_t stream);

size_t umma_score_workspace_bytes(int64_t B, int64_t C, int K);
bool umma_supported(int64_t B, int64_t C, int64_t D, int K);
// grid_share: batches meant to run at the same time (HGR_IMPL_GRID_SHARE); 1 = the whole grid
int umma_grid_share(int64_t B, int64_t C);
void umma_plan(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* plan);
int umma_footprint(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* out);
// C_total > 0 (with scatter->emit_bound): the lists are sized for a row's GLOBAL stream of C_total classes, of which
// this bank is one shard -- no local certificate / repair, the owner of the row certifies against the global K-th value
int launch_score_topk_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                           int32_t id_base, const int32_t* targets, int64_t B, int64_t C, int64_t D,
                           float scale, int K, void* ws, size_t ws_bytes, float* topk_val,
                           int32_t* topk_idx, int64_t* hits, int variant, bool skip_merge,
                           cudaStream_t stream, const OutScatter* scatter = nullptr, int64_t C_total = 0,
                           int grid_share = 1);
int umma_global_list_len(int64_t B, int64_t C, int64_t D, int K, int64_t C_total);
size_t umma_split_workspace_bytes(int64_t B, const Groups& gr, int K);
// scatter (class shard of the union bank, hgr_score_topk_splits_scatter_bounded): lists sized for each split's GLOBAL
// stream of split_C_total[s] classes; per split the local top-K and the bound of what was dropped go to the row owners,
// split s at + s * split_stride, instead of topk_val / topk_idx / counts
int launch_score_topk_splits_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                                  int32_t id_base, const int32_t* targets, const uint8_t* node_splits, int64_t n_nodes,
                                  int64_t B, int64_t C, int64_t D, float scale, int K, const Groups& gr,
                                  const uint8_t* group_splits, int S, void* ws, size_t ws_bytes, float* topk_val,
                                  int32_t* topk_idx, int64_t* counts, bool exact, cudaStream_t stream,
                                  const OutScatter* scatter = nullptr, const int64_t* split_C_total = nullptr,
                                  int64_t split_stride = 0);
int umma_split_global_list_len(int64_t B, int64_t C, int64_t D, int K, const Groups& gr, const uint8_t* group_splits,
                               int S, const int64_t* split_C_total);

int launch_level_argmax_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank_sorted, int64_t B, int64_t M, int64_t D,
                             const int32_t* level_end, int n_levels, unsigned long long* lvl_best, cudaStream_t stream);
// TOR / POR finish: node_splits NULL -> counts [HGR_HIER_MAX_CHAIN + 1][4]; otherwise counts [n_sets][...], a row
// added to set s for every bit s of node_splits[targets[row]]
int launch_hier_finish_rows(unsigned long long* lvl_best, int64_t B, int64_t M, int n_levels, const int32_t* sorted_to_pos,
                            const int32_t* first_out, const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                            const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits, int n_sets,
                            int32_t* lvl_idx, int32_t* top1, int64_t* counts, cudaStream_t stream);
// class-sharded TOR / POR (hgr_hier_level_scatter / hgr_hier_finish_rows_gathered)
int launch_hier_push(unsigned long long* lvl_best, int64_t B, int n_levels, int64_t row_base, int64_t block_rows,
                     int n_blocks, unsigned long long* const* dst, cudaStream_t stream);
int launch_hier_finish_gathered(const unsigned long long* parts, int n_parts, int64_t part_stride, int64_t B, int64_t M,
                                int n_levels, const int32_t* sorted_to_pos, const int32_t* first_out,
                                const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                                const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits,
                                int n_sets, int32_t* lvl_idx, int32_t* top1, int64_t* counts, cudaStream_t stream);
int launch_hier_mistakes(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets,
                         const int32_t* targets, const uint8_t* node_splits, const int32_t* chain_ptr,
                         const int32_t* chain_node, int64_t n_nodes, int64_t* counts, cudaStream_t stream);
// per-class Hit@k: counts [n_sets][n_nodes][HGR_NUM_HITS + 1] (class_hits.cu)
int launch_class_hits(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                      const uint8_t* node_splits, int64_t n_nodes, int64_t* counts, cudaStream_t stream);
int launch_normalize_dual(const void* E, int e_dtype, int64_t n_rows, int64_t D, void* out, const int32_t* dst_map,
                          void* out2, cudaStream_t stream);
// {threads, registers per thread, static shared memory, dynamic shared memory} of the row normalise of [*, D] rows
// of type e_dtype into bf16 (hgr_aggregate_normalize with identity CSR)
int normalize_rows_footprint(int e_dtype, int64_t D, int32_t* out);
int launch_normalize_bcast(const void* E, int e_dtype, int64_t n_rows, int64_t D, int64_t row0, int n_dst,
                           void* const* dst, cudaStream_t stream);

// cross-GPU sequencing of the peer-memory exchange (topk_merge.cu)
int launch_peer_signal(uint32_t* const* flags, int n, uint32_t* seq, cudaStream_t stream);
int launch_peer_wait(const uint32_t* flags, int n, uint32_t* seq, cudaStream_t stream);
int launch_logits_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, int64_t B, int64_t C,
                       int64_t D, float scale, float* out, int64_t ldo, cudaStream_t stream);

size_t masked_ce_workspace_bytes(int64_t B, int64_t U, int64_t T);
int launch_masked_ce(const float* logits, int64_t ldl, int64_t B, int64_t U, const int32_t* set_ptr,
                     const int32_t* set_col, const int32_t* label_pos, const float* weight, int64_t T,
                     float* loss, float* dlogits, void* ws, size_t ws_bytes, cudaStream_t stream);

size_t om_backward_workspace_bytes(int64_t B, int64_t U, int64_t D);
int launch_om_backward(const float* dlogits, const float* logits, int64_t ldl, int64_t B, int64_t U, int64_t D,
                       const __nv_bfloat16* x, const float* x_norm, const __nv_bfloat16* tn, const float* t_norm,
                       float scale, float* d_img, float* d_text, float* d_log_scale, void* ws, size_t ws_bytes,
                       cudaStream_t stream);

}  // namespace hgr
