// Hierarchical mistake severity and LCA distance@k (Bertinetto et al., "Making Better Mistakes", CVPR 2020) of the
// top-K lists the evaluator already holds on the device.  It extends the Hit@k count of the reference's test()
// (main.py:135-148): where that asks "is the label within the first k", this asks "how far from the label in the
// hierarchy are the first k".
//
// chain(n) = c2p[n] + [n] (chain table CSR over all nodes, evaluate.chain_csr); depth(n) = len(c2p[n]).  Every c2p[n]
// is a shortest root path (hierarchy.py), so the entry at index i of any chain has depth i, and a node common to two
// chains sits at the same index in both: lca(t, p) = the LARGEST index i with chain(t)[i] == chain(p)[i] (on a DAG the
// chains may split and join again), -1 (a virtual super-root) without one.
//   h(t, p) = depth(t) - depth(lca)            d(t, p) = depth(t) + depth(p) - 2 depth(lca)
// An empty list entry (id outside [0, n_nodes), e.g. -1 when C < K) counts as the super-root: h = d = depth(t) + 1.
//
// One warp per row.  Lane i holds chain(t)[i] (chain lengths <= HGR_HIER_MAX_CHAIN = 32); lane j first loads list entry
// j and its chain bounds, so the K chains' bounds arrive in one round.  Per entry, lane i loads chain(p)[i] and ONE
// ballot of equality gives the lca index (31 - clz).  The LCA lies at an index <= depth(t) <= 31 even when p is deeper,
// so 32 lanes always suffice; only d can exceed 2 * HGR_HIER_MAX_CHAIN and goes to the overflow bin.  All counts are
// warp-uniform: lane 0 adds them to the block's shared counters, one global atomic per non-zero counter and block.
#include "common.cuh"

namespace hgr {
namespace {

static_assert(HGR_HIER_MAX_CHAIN <= 32, "hier_mistakes matches a chain in one warp");
static_assert(HGR_TOPK_MAX <= 32, "hier_mistakes loads one list entry per lane");

constexpr int kMistakeRowsPerBlock = 8;
constexpr int kSumH = 2;                                   // slots 2..6: sum of h over the first min(k, K) entries
constexpr int kSumD = kSumH + HGR_NUM_HITS;                // slots 7..11: the same for d
constexpr int kHist = kSumD + HGR_NUM_HITS;                // slots 12..: histogram of d(t, p_0)
constexpr int kHistBins = 2 * HGR_HIER_MAX_CHAIN + 1;      // d = 0 .. 2 * HGR_HIER_MAX_CHAIN, then the overflow bin
static_assert(kHist + kHistBins + 1 == HGR_MISTAKE_COUNTERS, "counter layout of hgr_hier_mistakes");

__global__ void __launch_bounds__(kMistakeRowsPerBlock * 32)
hier_mistakes_kernel(const int32_t* __restrict__ topk_idx, int64_t B, int K, int64_t set_stride, int n_sets,
                     const int32_t* __restrict__ targets, const uint8_t* __restrict__ node_splits,
                     const int32_t* __restrict__ chain_ptr, const int32_t* __restrict__ chain_node, int64_t n_nodes,
                     unsigned long long* __restrict__ counts) {
  // 64-bit: a prediction's depth is not bounded by HGR_HIER_MAX_CHAIN, so neither is a block's sum of d
  __shared__ unsigned long long s_cnt[kMaxSplits * HGR_MISTAKE_COUNTERS];
  for (int i = threadIdx.x; i < n_sets * HGR_MISTAKE_COUNTERS; i += blockDim.x) s_cnt[i] = 0ull;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMistakeRowsPerBlock + (threadIdx.x >> 5);
  int32_t t = -1;
  int Lt = 0;
  if (row < B) {                                           // warp-uniform
    t = targets[row];
    if (t >= 0 && t < n_nodes) {
      Lt = chain_ptr[t + 1] - chain_ptr[t];
      if (Lt < 1 || Lt > HGR_HIER_MAX_CHAIN) Lt = 0;
    }
  }
  if (Lt > 0) {                                            // warp-uniform: the row counts
    const int dt = Lt - 1;
    const int32_t ct = lane < Lt ? chain_node[chain_ptr[t] + lane] : -2;
    const unsigned bits = node_splits ? node_splits[t] : 1u;
    for (int s = 0; s < n_sets; ++s) {
      if (!((bits >> s) & 1u)) continue;
      // lane j: list entry j and its chain [c0, c0 + Lp); Lp = 0 for an empty entry
      int32_t pj = -1, c0 = 0, Lp = 0;
      if (lane < K) {
        pj = topk_idx[s * set_stride + row * K + lane];
        if (pj >= 0 && pj < n_nodes) {
          c0 = chain_ptr[pj];
          Lp = chain_ptr[pj + 1] - c0;
        }
      }
      unsigned h_sum[HGR_NUM_HITS] = {};
      unsigned long long d_sum[HGR_NUM_HITS] = {};
      int d0 = 0;
      for (int j = 0; j < K; ++j) {
        const int32_t pc0 = __shfl_sync(0xffffffffu, c0, j);
        const int32_t lp = __shfl_sync(0xffffffffu, Lp, j);
        int h, d;
        if (lp > 0) {
          const int32_t cp = lane < lp ? chain_node[pc0 + lane] : -3;
          const unsigned m = __ballot_sync(0xffffffffu, cp == ct);   // ct = -2 past the label's chain
          const int lca = m ? 31 - __clz(m) : -1;
          h = dt - lca;
          d = dt + (lp - 1) - 2 * lca;
        } else {
          h = d = dt + 1;                                  // empty entry: the super-root
        }
        if (j == 0) d0 = d;
#pragma unroll
        for (int c = 0; c < HGR_NUM_HITS; ++c)
          if (j < hit_cut(c)) {
            h_sum[c] += h;
            d_sum[c] += d;
          }
      }
      if (lane == 0) {                                     // lane 0 holds entry 0
        unsigned long long* c = s_cnt + s * HGR_MISTAKE_COUNTERS;
        atomicAdd(c + 0, 1ull);
        if (pj != t) atomicAdd(c + 1, 1ull);
#pragma unroll
        for (int k = 0; k < HGR_NUM_HITS; ++k) {
          if (h_sum[k]) atomicAdd(c + kSumH + k, static_cast<unsigned long long>(h_sum[k]));
          if (d_sum[k]) atomicAdd(c + kSumD + k, d_sum[k]);
        }
        atomicAdd(c + kHist + (d0 < kHistBins ? d0 : kHistBins), 1ull);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_sets * HGR_MISTAKE_COUNTERS; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(counts + i, s_cnt[i]);
}

}  // namespace

int launch_hier_mistakes(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets,
                         const int32_t* targets, const uint8_t* node_splits, const int32_t* chain_ptr,
                         const int32_t* chain_node, int64_t n_nodes, int64_t* counts, cudaStream_t stream) {
  const int blocks = static_cast<int>((B + kMistakeRowsPerBlock - 1) / kMistakeRowsPerBlock);   // one warp per row
  hier_mistakes_kernel<<<blocks, kMistakeRowsPerBlock * 32, 0, stream>>>(
      topk_idx, B, K, set_stride, n_sets, targets, node_splits, chain_ptr, chain_node, n_nodes,
      reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
