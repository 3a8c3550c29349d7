// Per-class Hit@{1,2,5,10,20} of the top-K lists the evaluator already holds on the device: the reference's Hit@k
// (main.py:135-148) counted per label, so that the class-averaged accuracy of the zero-shot literature (e.g. Xian et al.,
// TPAMI 2018) can be derived.  counts[s][t] = {Hit@1, Hit@2, Hit@5, Hit@10, Hit@20, rows} of the rows labelled t in list
// set s: the layout of the per-split counters of hgr_score_topk_splits, one row per class.
//
// One thread per row scans the first min(K, 20) entries of its list for its label (first match, the rule of finish_row /
// count_split_row in topk_merge.cu); positions past 20 count toward no Hit@k.  The reference's test loader puts one class
// in a batch, so the rows of a warp mostly share one label and so one counter row: __match_any_sync groups the lanes of
// equal label, one ballot per Hit@k cut gives every group's counts by popcount, and the group's lowest lane adds the
// non-zero ones -- at most HGR_NUM_HITS + 1 global atomics per label and warp, never one per row.
#include "common.cuh"

namespace hgr {
namespace {

constexpr int kClassHitsThreads = 128;
constexpr int kClassHitsScan = hit_cut(HGR_NUM_HITS - 1);   // entries that can count toward some Hit@k

__global__ void __launch_bounds__(kClassHitsThreads)
class_hits_kernel(const int32_t* __restrict__ topk_idx, int64_t B, int K, int64_t set_stride, int n_sets,
                  const int32_t* __restrict__ targets, const uint8_t* __restrict__ node_splits, int64_t n_nodes,
                  unsigned long long* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kClassHitsThreads + threadIdx.x;
  int32_t t = -1;
  unsigned bits = 0u;                                      // the list sets this row counts in
  if (row < B) {
    t = targets[row];
    if (t >= 0 && t < n_nodes) bits = node_splits ? node_splits[t] : 1u;
  }
  const int scan = K < kClassHitsScan ? K : kClassHitsScan;
  for (int s = 0; s < n_sets; ++s) {                       // every lane runs every set: the warp votes below
    const bool counts_here = (bits >> s) & 1u;
    int pos = kClassHitsScan;                              // past every cut: no hit
    if (counts_here) {
      const int32_t* list = topk_idx + s * set_stride + row * K;
#pragma unroll
      for (int j = kClassHitsScan - 1; j >= 0; --j)        // independent loads, all in flight; the lowest match wins
        if (j < scan && list[j] == t) pos = j;
    }
    // lanes of one label (and counting in set s) form one group; the others share the key -1 and are never flushed
    const unsigned group = __match_any_sync(0xffffffffu, counts_here ? t : -1);
    unsigned hit[HGR_NUM_HITS];
#pragma unroll
    for (int c = 0; c < HGR_NUM_HITS; ++c) hit[c] = __ballot_sync(0xffffffffu, pos < hit_cut(c)) & group;
    if (counts_here && lane == __ffs(group) - 1) {
      unsigned long long* cnt = counts + (static_cast<int64_t>(s) * n_nodes + t) * (HGR_NUM_HITS + 1);
#pragma unroll
      for (int c = 0; c < HGR_NUM_HITS; ++c)
        if (hit[c]) atomicAdd(cnt + c, static_cast<unsigned long long>(__popc(hit[c])));
      atomicAdd(cnt + HGR_NUM_HITS, static_cast<unsigned long long>(__popc(group)));
    }
  }
}

}  // namespace

int launch_class_hits(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                      const uint8_t* node_splits, int64_t n_nodes, int64_t* counts, cudaStream_t stream) {
  const int blocks = static_cast<int>((B + kClassHitsThreads - 1) / kClassHitsThreads);   // one thread per row
  class_hits_kernel<<<blocks, kClassHitsThreads, 0, stream>>>(topk_idx, B, K, set_stride, n_sets, targets, node_splits,
                                                             n_nodes, reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
