// Host side of kernel (2): TMA descriptors, the work split over the CTA pairs, the list-length policy and the launchers
// of hgr_score_topk / hgr_logits_dense.  The kernel itself is score_pair.cu; the merge of the per-worker lists is
// topk_merge.cu.
//
// Reference: `feats @ self.zsl_weights.T` (model/clip_tree.py:331), `logits[:, test_index]` +
// `.topk(20, 1, True, True)` (main.py:136-138), id mapping / hit test (main.py:139-147).
#include <cuda.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "sketch_epi.cuh"
#include "umma_common.cuh"

namespace hgr {
using namespace umma;
namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}

// [rows, D] row-major bf16 matrix, box = [box_rows, 64] elements, 128B swizzle, zero OOB fill
int make_map(CUtensorMap* map, const void* base, int64_t rows, int64_t D, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return set_error(HGR_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(D) * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(kBlockK), static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(HGR_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return HGR_OK;
}

// Columns per worker up to which a stream counts as short: per-segment and per-launch costs, not the main loop, decide
constexpr int64_t kShortStreamCols = 3072;
// Grid share the streaming evaluator asks for on short streams (umma_grid_share)
constexpr int kStreamGridShare = 2;

// CTA pairs the persistent kernel runs on
int usable_sms() {
  const int n = num_sms();
  return n < 2 ? 2 : n;
}

// Rough cost of the slowest worker of a schedule, in operand columns streamed through shared memory: every
// sub-tile re-streams the A operand (one row tile = 256 "columns" worth of bytes) next to its own bank rows, and
// every segment (row tile x worker intersection) starts a fresh list (floor pass, warm-up inserts, list write-out).
static double sched_cost(const Sched& s) {
  constexpr double kSegmentOverhead = 400.0;   // ~3-4 us of floor pass + warm-up inserts + list write-out
  double worst = 0.0;
  for (int32_t w = 0; w < s.G; ++w) {
    int64_t u = s.unit_begin(w);
    const int64_t u_end = s.unit_begin(w + 1);
    double cost = 0.0;
    while (u < u_end) {
      const int64_t tile_end = (u / s.U + 1) * s.U;
      const int64_t e = u_end < tile_end ? u_end : tile_end;
      const int64_t cols = (e - u) * kUnit;
      cost += static_cast<double>((cols + kSubN - 1) / kSubN) * 256.0 + static_cast<double>(cols) + kSegmentOverhead;
      u = e;
    }
    worst = cost > worst ? cost : worst;
  }
  return worst;
}

// Workers: all CTA pairs, unless a slightly smaller count that is a multiple of the row-tile count wins -- then no
// chunk straddles a row tile (one list per worker, no ragged sub-tiles at both ends; measured at B = 4096:
// 64 aligned pairs beat 74 for every bank size, e.g. 33.6 vs 39.7 us at C = 2,731).
//
// grid_share c > 1: the call is one of c batches meant to run side by side (the streaming evaluator's round-robin
// streams), so it takes floor(pairs / c) pairs, rounded down to a multiple of the row tiles.  Each worker then streams
// c times the columns: its fixed costs (set-up, first operands, exposed tail) and the A-operand re-stream of its
// remainder sub-tile are paid once per longer run, and a row has fewer, longer lists.
Sched pick_sched(int64_t B, int64_t C, int grid_share = 1) {
  const int most = usable_sms() / 2;
  if (grid_share > 1) {
    const int budget = most / grid_share > 0 ? most / grid_share : 1;
    const int MT = static_cast<int>((B + 2 * kTileM - 1) / (2 * kTileM));
    return make_sched(B, C, budget >= MT ? budget / MT * MT : budget, 2 * kTileM);
  }
  Sched best = make_sched(B, C, most, 2 * kTileM);
  if (best.MT > 1 && best.MT <= most && best.G == most) {
    const int aligned = most / best.MT * best.MT;
    if (aligned != most && aligned * 10 >= most * 8) {
      const Sched alt = make_sched(B, C, aligned, 2 * kTileM);
      // only for short streams (<= kShortStreamCols columns per worker): there the per-segment costs decide; on long
      // streams the fewer, larger lists of the aligned split sit closer to the speculation limit (an expected repair
      // of a 5,000-column range costs more than the alignment saves -- measured at cfg 5)
      const int64_t cols_per_worker = (alt.T + alt.G - 1) / alt.G * kUnit;
      if (cols_per_worker <= kShortStreamCols && sched_cost(alt) < sched_cost(best)) best = alt;
    }
  }
  return best;
}

int common_setup(const __nv_bfloat16* X, const __nv_bfloat16* bank, int64_t B, int64_t C, int64_t D,
                 CUtensorMap* mx, CUtensorMap* mb, Params* p, int grid_share = 1) {
  int rc = make_map(mx, X, B, D, kTileM);
  if (rc != HGR_OK) return rc;
  rc = make_map(mb, bank, C, D, kBBoxRows);
  if (rc != HGR_OK) return rc;
  p->sched = pick_sched(B, C, grid_share);
  p->B = B;
  p->C = C;
  p->num_k_blocks = static_cast<int>((D + kBlockK - 1) / kBlockK);
  return HGR_OK;
}

// ---- list-width policy -------------------------------------------------------------------
// With bank rows in random order, each of a row's true top-K members falls into a given list with probability
// `share` = the fraction of the row's columns that list streams (the largest one: a worker's chunk of the schedule).
// A list of KL < K entries cannot be certified when it receives KL or more of them: probability <= C(K, KL) *
// share^KL.  A repair re-scans that list's column range with ONE warp of the merge kernel: measured ~0.6 us per bank
// row of 1024 elements (a 590-column range of cfg 2: 0.36 ms; a 4,700-column range of cfg 5: 2.8 ms), and the whole
// call waits for it.
double overflow_bound(int K, int KL, double share) {
  double c = 1.0;
  for (int i = 0; i < KL; ++i) c = c * (K - i) / (i + 1);
  return c * std::pow(share, KL);
}

double max_list_share(const Sched& s) {
  const double chunk = static_cast<double>((s.T + s.G - 1) / s.G);   // units per worker
  const double share = chunk / static_cast<double>(s.U);
  return share > 1.0 ? 1.0 : share;
}

// Speculate only while the EXPECTED repair time per call stays below 1.5 % of the call's estimated duration (main
// loop at 60 % of the bf16 peak).  cfg 2 (37 lists of 590 columns per row, KL = 8): 7e-4 repairs x 0.36 ms = 0.25 us
// of 24 us -- accepted, and worth it (exact 20-entry lists cost 55 us there).  cfg 2 on half the grid (grid share 2: 18
// lists of 1,216 columns): KL = 8 expects 0.1 repairs per call, KL = 10 5e-4 -- KL = 10.  B = 4096 (4-6 lists per row):
// 16-entry lists would save ~6 us per call but cost 1-8 us in expected repairs -- rejected, exact lists run in the same
// deferred-insert mode.
int pick_list_len(int K, int64_t B, int64_t C, int64_t D, int lists_per_row, double share, bool allow_speculation) {
  const int exact = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  if (!allow_speculation) return exact;
#ifdef HGR_FORCE_KL   // kernel experiments (tools/build_variant.sh): the list length the policy is NOT allowed to pick
  if (HGR_FORCE_KL < K) return HGR_FORCE_KL;
#endif
  const int cand[4] = {8, 10, 12, 16};
  for (int i = 0; i < 4; ++i) {
    const int kl = cand[i];
    if (kl >= K) break;
    const double repairs = static_cast<double>(B) * lists_per_row * overflow_bound(K, kl, share);
    const double t_repair = share * static_cast<double>(C) * (static_cast<double>(D) / 1024.0) * 0.6e-6;
    const double t_call = 2.0 * static_cast<double>(B) * static_cast<double>(C) * static_cast<double>(D) / (0.6 * 1.6e15);
    if (repairs * t_repair < 0.015 * t_call) return kl;
  }
  return exact;
}

// Class shard of a row's GLOBAL stream (hgr_score_topk_scatter_bounded): the certificate is taken by the owner of the
// row against the global K-th value, so what counts is the share of the GLOBAL stream one list holds, and a repair
// re-scans the doubtful shard completely with one warp, possibly over NVLink (budgeted at 1.5 us per bank row of 1024
// elements).  N = 8 (4 lists of 683 of 21,841 columns per row and rank): KL = 10, 2e-5 repairs per batch; N = 4:
// KL = 12; N = 2: KL = 16.
int pick_list_len_global(int K, int64_t B, int64_t C, int64_t D, int64_t C_total, const Sched& s) {
  const int exact = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  if (C_total < C) C_total = C;
  const double cols = static_cast<double>((s.T + s.G - 1) / s.G) * kUnit;           // columns of the largest list
  const double share = cols / static_cast<double>(C_total) > 1.0 ? 1.0 : cols / static_cast<double>(C_total);
  const double lists = static_cast<double>(s.P) * static_cast<double>(C_total) / static_cast<double>(C);
  const int cand[4] = {8, 10, 12, 16};
  for (int i = 0; i < 4; ++i) {
    const int kl = cand[i];
    if (kl >= K) break;
    const double repairs = static_cast<double>(B) * lists * overflow_bound(K, kl, share);
    const double t_repair = static_cast<double>(C) * (static_cast<double>(D) / 1024.0) * 1.5e-6;
    const double t_call = 2.0 * static_cast<double>(B) * static_cast<double>(C) * static_cast<double>(D) / (0.6 * 1.6e15);
    if (repairs * t_repair < 0.015 * t_call) return kl;
  }
  return exact;
}

}  // namespace

int umma_global_list_len(int64_t B, int64_t C, int64_t D, int K, int64_t C_total) {
  return pick_list_len_global(K, B, C, D, C_total, pick_sched(B, C));
}

// floor-sketch epilogue: [B][20] floor words, [P][B] list lengths, [P][B][kSkCap] (value, bank row) entries
static size_t sketch_workspace_bytes(int64_t B, int P) {
  return static_cast<size_t>(B) * kSkSlots * 8 + static_cast<size_t>(P) * B * 4 + static_cast<size_t>(P) * B * kSkCap * 8 + 64;
}

bool umma_supported(int64_t B, int64_t C, int64_t D, int K) {
  return B >= 1 && C >= 1 && D >= 8 && D % 8 == 0 && K >= 1 && K <= HGR_TOPK_MAX &&
         C < (int64_t(1) << 31) - 512 && B < (int64_t(1) << 31) - 512;
}

size_t umma_score_workspace_bytes(int64_t B, int64_t C, int K) {
  // worst case over the grid shares, the list-width policy (exact lists) and the candidate lists of the floor-sketch
  // variant (all pairs)
  int p2 = 1;
  for (int c = 1; c <= HGR_GRID_SHARE_MAX; ++c) {
    const int p = pick_sched(B, C, c).P;
    p2 = p > p2 ? p : p2;
  }
  const int p4 = make_sched(B, C, usable_sms() / 2, 2 * kTileM).P;
  const int kl = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  const size_t lists = static_cast<size_t>(p2) * B * kl * (sizeof(float) + sizeof(int32_t));
  const size_t sketch = sketch_workspace_bytes(B, p4 > p2 ? p4 : p2);
  return (lists > sketch ? lists : sketch) + kWsHeaderBytes;
}

// The grid share for a batch that runs beside others (the streaming evaluator): on short streams (<= kShortStreamCols
// columns per worker on the whole grid) kStreamGridShare, the best of shares 1-4 measured at cfg 2
// (profiles/r09_concurrent_grid); long streams (every B >= 2048, e.g. cfg 5) keep the schedule of a lone call.
int umma_grid_share(int64_t B, int64_t C) {
  if (B >= 2048) return 1;
  const Sched s = pick_sched(B, C);
  return (s.T + s.G - 1) / s.G * kUnit <= kShortStreamCols ? kStreamGridShare : 1;
}

// The decisions launch_score_topk_umma takes for the production variant, without launching anything.
void umma_plan(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* plan) {
  const Sched s = pick_sched(B, C, grid_share);
  plan[0] = s.G;
  plan[1] = s.MT;
  plan[2] = s.U;
  plan[3] = s.P;
  plan[4] = pick_list_len(K, B, C, D, s.P, max_list_share(s), true);
  plan[5] = 1;
  plan[6] = pair_ring_depth(B);
  plan[7] = static_cast<int32_t>((s.T + s.G - 1) / s.G * kUnit);
}

// The production scoring kernel and the merge behind it as launch_score_topk_umma runs them: {threads, registers per
// thread, static shared memory, dynamic shared memory} of each.
int umma_footprint(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* out) {
  int32_t plan[8];
  umma_plan(B, C, D, K, grid_share, plan);
  const int rc = pair_kernel_footprint(B, plan[4], out);
  return rc != HGR_OK ? rc : merge_kernel_footprint(plan[3], plan[4], out + 4);
}

int launch_score_topk_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                           int32_t id_base, const int32_t* targets, int64_t B, int64_t C, int64_t D, float scale,
                           int K, void* ws, size_t ws_bytes, float* topk_val, int32_t* topk_idx, int64_t* hits,
                           int variant, bool skip_merge, cudaStream_t stream, const OutScatter* scatter,
                           int64_t C_total, int grid_share) {
  // variants: kVarProd   production: deferred-insert lists, speculative (KL < K) when provably cheap
  //           kVarExact  the same kernel with K-entry lists (no speculation)
  //           kVarNull   main loop with a trivial epilogue (ceiling; NOT a top-k) -- diagnostics only
  //           kVarSketch floor-sketch epilogue (sketch_epi.cuh): exact, independent of the bank order
  if (ws == nullptr || ws_bytes < umma_score_workspace_bytes(B, C, K))
    return set_error(HGR_ERR_WORKSPACE, "hgr_score_topk(tcgen05): workspace %zu < %zu bytes", ws_bytes,
                     umma_score_workspace_bytes(B, C, K));
  CUtensorMap mx, mb;
  Params p{};
  int rc = common_setup(X, bank, B, C, D, &mx, &mb, &p, grid_share);
  if (rc != HGR_OK) return rc;
  p.scale = scale;
  p.stats = static_cast<unsigned int*>(ws);                              // header: statistics, timeline stamps
  static const bool want_timeline = getenv("HGR_TIMELINE") != nullptr;   // diagnostics (tools/timeline.py)
  p.timeline = want_timeline ? reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(ws) + 64) : nullptr;
  MergeArgs m{};
  if (variant == kVarSketch) {
    if (K > kSkKeep) return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk(tcgen05 sketch): K = %d > %d", K, kSkKeep);
    p.sched = make_sched(B, C, usable_sms() / 2, 2 * kTileM);   // lists are cheap here: every pair works
    uint8_t* w = static_cast<uint8_t*>(ws) + kWsHeaderBytes;
    p.sk_floors = reinterpret_cast<unsigned long long*>(w);
    w += static_cast<size_t>(B) * kSkSlots * 8;
    p.sk_part = reinterpret_cast<uint2*>(w);
    w += static_cast<size_t>(p.sched.P) * B * kSkCap * 8;
    p.sk_cnt = reinterpret_cast<int32_t*>(w);
    rc = launch_pair_kernel(kEpiSketch, 8, mx, mb, p, stream);
    m.sk_part = p.sk_part;
    m.sk_cnt = p.sk_cnt;
    m.sk_cap = kSkCap;
    m.KL = K;
  } else {
    const bool global_cert = variant == kVarProd && C_total > 0 && scatter != nullptr && scatter->emit_bound != 0;
    const int KL = global_cert ? pick_list_len_global(K, B, C, D, C_total, p.sched)
                               : pick_list_len(K, B, C, D, p.sched.P, max_list_share(p.sched), variant == kVarProd);
    p.KL = KL;
    p.part_val = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes);
    p.part_idx = reinterpret_cast<int32_t*>(p.part_val + static_cast<size_t>(p.sched.P) * B * KL);
    if (variant == kVarNull) return launch_pair_kernel(kEpiNull, 8, mx, mb, p, stream);
    rc = launch_pair_kernel(kEpiTopkDefer, KL, mx, mb, p, stream);
    m.part_val = p.part_val;
    m.part_idx = p.part_idx;
    m.KL = KL;
    m.X = X;
    m.bank = bank;
    m.D8 = static_cast<int>(D / 8);
    m.rescan_count = p.stats;
  }
  if (rc != HGR_OK || skip_merge) return rc;
  m.P = p.sched.P;
  m.B = B;
  m.K = K;
  m.use_sched = 1;
  m.sched = p.sched;
  m.col_id = col_id;
  m.id_base = id_base;
  m.scale = scale;
  m.targets = targets;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  m.hits = hits;
  m.C = C;
  if (scatter) m.scatter = *scatter;
  return launch_topk_merge(m, stream);
}

// ---- several test splits in one pass (hgr_score_topk_splits) --------------------------------------------------------
// Grouped schedule over all workers (sched.cuh): no list crosses a group, so split s is served by the lists of its
// groups alone.  The list length comes from the split that is worst off: for split s a list holds at most `cols_s` of
// its C_s columns (share_s = cols_s / C_s), and each row has `lists_s` lists of s; the narrowest length whose expected
// repair time stays below 1.5 % of the call (the rule of pick_list_len, the call being the GEMM over all C columns)
// for EVERY split is taken -- so a small split covered by a few long lists per row does not get repaired on every row.

// Per split: its columns in this bank (cs), the columns of its largest list (cols) and the most lists of it a row has.
struct SplitStats {
  int64_t cs[kMaxSplits] = {}, cols[kMaxSplits] = {};
  int lists[kMaxSplits] = {};
};

static SplitStats split_stats(const Sched& s, const Groups& gr, const uint8_t* group_splits, int S) {
  SplitStats st;
  for (int g = 0; g < gr.n; ++g)
    for (int sp = 0; sp < S; ++sp)
      if ((group_splits[g] >> sp) & 1u) st.cs[sp] += gr.end[g] - gr.begin(g);
  for (int32_t mt = 0; mt < s.MT; ++mt) {
    int n[kMaxSplits] = {};
    const int parts = group_parts(s, gr, mt);
    for (int p = 0; p < parts; ++p) {
      int64_t c0, c1;
      const int g = group_slot_range(s, gr, mt, p, c0, c1);
      for (int sp = 0; sp < S; ++sp) {
        if (!((group_splits[g] >> sp) & 1u)) continue;
        ++n[sp];
        st.cols[sp] = c1 - c0 > st.cols[sp] ? c1 - c0 : st.cols[sp];
      }
    }
    for (int sp = 0; sp < S; ++sp) st.lists[sp] = n[sp] > st.lists[sp] ? n[sp] : st.lists[sp];
  }
  return st;
}

static int pick_list_len_splits(int K, int64_t B, int64_t C, int64_t D, const Sched& s, const Groups& gr,
                                const uint8_t* group_splits, int S) {
  const int exact = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  const SplitStats st = split_stats(s, gr, group_splits, S);
  const int64_t* cs = st.cs;
  const int64_t* cols = st.cols;
  const int* lists = st.lists;
  const double t_call = 2.0 * static_cast<double>(B) * static_cast<double>(C) * static_cast<double>(D) / (0.6 * 1.6e15);
  const int cand[4] = {8, 10, 12, 16};
  for (int i = 0; i < 4; ++i) {
    const int kl = cand[i];
    if (kl >= K) break;
    bool ok = true;
    for (int sp = 0; sp < S && ok; ++sp) {
      if (cs[sp] == 0) continue;
      const double share = static_cast<double>(cols[sp]) / static_cast<double>(cs[sp]);
      const double repairs = static_cast<double>(B) * lists[sp] * overflow_bound(K, kl, share);
      const double t_repair = static_cast<double>(cols[sp]) * (static_cast<double>(D) / 1024.0) * 0.6e-6;
      ok = repairs * t_repair < 0.015 * t_call;
    }
    if (ok) return kl;
  }
  return exact;
}

// Class shard of the union bank (hgr_score_topk_splits_scatter_bounded): the certificate of split s is taken by the row
// owner against s's GLOBAL K-th value, so -- as pick_list_len_global does for one bank -- a list's share is its columns
// over the split's global class count split_C_total[s], a row has lists_s * split_C_total[s] / cs_s lists of s over all
// ranks, and a repair re-scans s's rows of one shard (budgeted at 1.5 us per bank row of 1024 elements, NVLink).  The
// narrowest length whose expected repair time stays below 1.5 % of this rank's GEMM for every split is taken.
static int pick_list_len_splits_global(int K, int64_t B, int64_t C, int64_t D, const Sched& s, const Groups& gr,
                                       const uint8_t* group_splits, int S, const int64_t* split_C_total) {
  const int exact = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  const SplitStats st = split_stats(s, gr, group_splits, S);
  const double t_call = 2.0 * static_cast<double>(B) * static_cast<double>(C) * static_cast<double>(D) / (0.6 * 1.6e15);
  const int cand[4] = {8, 10, 12, 16};
  for (int i = 0; i < 4; ++i) {
    const int kl = cand[i];
    if (kl >= K) break;
    bool ok = true;
    for (int sp = 0; sp < S && ok; ++sp) {
      if (st.cs[sp] == 0) continue;
      const double total = static_cast<double>(split_C_total[sp] > st.cs[sp] ? split_C_total[sp] : st.cs[sp]);
      const double share = static_cast<double>(st.cols[sp]) / total > 1.0 ? 1.0 : static_cast<double>(st.cols[sp]) / total;
      const double lists = static_cast<double>(st.lists[sp]) * total / static_cast<double>(st.cs[sp]);
      const double repairs = static_cast<double>(B) * lists * overflow_bound(K, kl, share);
      const double t_repair = static_cast<double>(st.cs[sp]) * (static_cast<double>(D) / 1024.0) * 1.5e-6;
      ok = repairs * t_repair < 0.015 * t_call;
    }
    if (ok) return kl;
  }
  return exact;
}

// The schedule and the list length of a call depend only on (B, C, D, K, group table, split bits) and visit every
// (row tile, slot): eager callers (evaluate.test, SplitEval.update) make the same call every batch, so the last few
// plans are kept.
struct SplitPlan {
  int64_t B = -1, C = -1, D = -1;
  int K = 0, S = 0;
  bool exact = false;
  Groups gr{};
  uint8_t splits[kMaxGroups] = {};
  int64_t ctot[kMaxSplits] = {};   // global class count of every split (class shard), all 0 otherwise
  Sched sched{};
  int KL = 0;
};

static SplitPlan split_plan(int64_t B, int64_t C, int64_t D, int K, const Groups& gr, const uint8_t* group_splits, int S,
                            bool exact, const int64_t* split_C_total = nullptr) {
  constexpr int kSlots = 8;
  static SplitPlan cache[kSlots];
  static int next = 0;
  static std::mutex mu;
  SplitPlan key;
  key.B = B, key.C = C, key.D = D, key.K = K, key.S = S, key.exact = exact;
  key.gr = gr;
  for (int g = 0; g < gr.n && group_splits; ++g) key.splits[g] = group_splits[g];
  for (int sp = 0; sp < S && split_C_total; ++sp) key.ctot[sp] = split_C_total[sp];
  auto same = [&](const SplitPlan& e) {
    return e.B == key.B && e.C == key.C && e.D == key.D && e.K == key.K && e.S == key.S && e.exact == key.exact &&
           std::memcmp(&e.gr, &key.gr, sizeof(Groups)) == 0 && std::memcmp(e.splits, key.splits, kMaxGroups) == 0 &&
           std::memcmp(e.ctot, key.ctot, sizeof(key.ctot)) == 0;
  };
  {
    std::lock_guard<std::mutex> lk(mu);
    for (const SplitPlan& e : cache)
      if (same(e)) return e;
  }
  key.sched = make_sched_groups(B, gr, usable_sms() / 2, 2 * kTileM);
  const int exact_kl = K <= 8 ? 8 : (K <= 12 ? 12 : (K <= 20 ? 20 : 32));
  key.KL = exact || group_splits == nullptr ? exact_kl
           : split_C_total ? pick_list_len_splits_global(K, B, C, D, key.sched, gr, group_splits, S, split_C_total)
                           : pick_list_len_splits(K, B, C, D, key.sched, gr, group_splits, S);
  std::lock_guard<std::mutex> lk(mu);
  cache[next] = key;
  next = (next + 1) % kSlots;
  return key;
}

size_t umma_split_workspace_bytes(int64_t B, const Groups& gr, int K) {
  // sized for exact lists: the plan without split bits (the list length does not change the schedule)
  const SplitPlan plan = split_plan(B, gr.end[gr.n - 1], 0, K, gr, nullptr, 0, true);
  return static_cast<size_t>(plan.sched.P) * B * plan.KL * (sizeof(float) + sizeof(int32_t)) + kWsHeaderBytes;
}

int launch_score_topk_splits_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, const int32_t* col_id,
                                  int32_t id_base, const int32_t* targets, const uint8_t* node_splits, int64_t n_nodes,
                                  int64_t B, int64_t C, int64_t D, float scale, int K, const Groups& gr,
                                  const uint8_t* group_splits, int S, void* ws, size_t ws_bytes, float* topk_val,
                                  int32_t* topk_idx, int64_t* counts, bool exact, cudaStream_t stream,
                                  const OutScatter* scatter, const int64_t* split_C_total, int64_t split_stride) {
  if (ws == nullptr || ws_bytes < umma_split_workspace_bytes(B, gr, K))
    return set_error(HGR_ERR_WORKSPACE, "%s: workspace %zu < %zu bytes",
                     scatter ? "hgr_score_topk_splits_scatter_bounded" : "hgr_score_topk_splits", ws_bytes,
                     umma_split_workspace_bytes(B, gr, K));
  CUtensorMap mx, mb;
  Params p{};
  int rc = common_setup(X, bank, B, C, D, &mx, &mb, &p);
  if (rc != HGR_OK) return rc;
  const SplitPlan plan = split_plan(B, C, D, K, gr, group_splits, S, exact, split_C_total);
  p.sched = plan.sched;
  p.groups = gr;
  p.scale = scale;
  p.stats = static_cast<unsigned int*>(ws);
  const int KL = plan.KL;
  p.KL = KL;
  p.part_val = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes);
  p.part_idx = reinterpret_cast<int32_t*>(p.part_val + static_cast<size_t>(p.sched.P) * B * KL);
  rc = launch_pair_kernel(kEpiTopkGroups, KL, mx, mb, p, stream);
  if (rc != HGR_OK) return rc;
  SplitMergeArgs m{};
  m.part_val = p.part_val;
  m.part_idx = p.part_idx;
  m.B = B;
  m.C = C;
  m.KL = KL;
  m.K = K;
  m.S = S;
  m.sched = p.sched;
  m.groups = gr;
  for (int g = 0; g < gr.n; ++g) m.group_splits[g] = group_splits[g];
  m.col_id = col_id;
  m.id_base = id_base;
  m.scale = scale;
  m.targets = targets;
  m.node_splits = node_splits;
  m.n_nodes = n_nodes;
  m.topk_val = topk_val;
  m.topk_idx = topk_idx;
  m.counts = counts;
  m.X = X;
  m.bank = bank;
  m.D8 = static_cast<int>(D / 8);
  m.rescan_count = p.stats;
  if (scatter) m.scatter = *scatter;
  m.split_stride = split_stride;
  return launch_topk_split_merge(m, stream);
}

int umma_split_global_list_len(int64_t B, int64_t C, int64_t D, int K, const Groups& gr, const uint8_t* group_splits,
                               int S, const int64_t* split_C_total) {
  return split_plan(B, C, D, K, gr, group_splits, S, false, split_C_total).KL;
}

// Row f1 without the dense matrix: X . bank_sorted^T on the tcgen05 loop, per-level arg-max in the epilogue.
int launch_level_argmax_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank_sorted, int64_t B, int64_t M, int64_t D,
                             const int32_t* level_end, int n_levels, unsigned long long* lvl_best, cudaStream_t stream) {
  if (n_levels < 1 || n_levels > kMaxHierLevels)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics_fused_rows / hgr_hier_level_scatter: %d levels outside [1, %d]",
                     n_levels, kMaxHierLevels);
  CUtensorMap mx, mb;
  Params p{};
  int rc = common_setup(X, bank_sorted, B, M, D, &mx, &mb, &p);
  if (rc != HGR_OK) return rc;
  p.KL = 0;
  p.scale = 1.f;
  p.n_levels = n_levels;
  int32_t prev = 0;
  for (int l = 0; l < n_levels; ++l) {
    if (level_end[l] < prev || level_end[l] > M)
      return set_error(HGR_ERR_BAD_ARG,
                       "hgr_hier_metrics_fused_rows / hgr_hier_level_scatter: level_end must be non-decreasing and <= M");
    p.lvl_end[l] = prev = level_end[l];
  }
  if (prev != M)
    return set_error(HGR_ERR_BAD_ARG, "hgr_hier_metrics_fused_rows / hgr_hier_level_scatter: level_end[n_levels - 1] must be M");
  // all zero: on first use by contract, afterwards because hier_finish_rows_kernel / hier_push_kernel zero what they read
  p.lvl_best = lvl_best;
  return launch_pair_kernel(kEpiLevel, 8, mx, mb, p, stream);
}

int launch_logits_umma(const __nv_bfloat16* X, const __nv_bfloat16* bank, int64_t B, int64_t C, int64_t D,
                       float scale, float* out, int64_t ldo, cudaStream_t stream) {
  CUtensorMap mx, mb;
  Params p{};
  int rc = common_setup(X, bank, B, C, D, &mx, &mb, &p);
  if (rc != HGR_OK) return rc;
  p.KL = 0;
  p.scale = scale;
  p.dense_out = out;
  p.ldo = ldo;
  return launch_pair_kernel(kEpiDense, 8, mx, mb, p, stream);
}

}  // namespace hgr
