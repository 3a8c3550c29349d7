// TOR / POR hierarchical metrics (reference main.py:143,152-191), second half of the fused path.
//
// Per batch the reference takes the arg-max over `train_index` (TOR, :155-160) and, for every node p of the label's
// ancestor chain, clones the [B, N] logits, fills every column that is not at p's depth with -1, gathers `train_index`
// and takes another arg-max (:163-176) -- L + 1 passes over B x N plus a Python B x L loop with device->host copies
// (:177-191).  Here the per-level arg-max over the train columns runs in the epilogue of the GEMM against the train
// rows of the bank sorted by level (score_pair.cu, kEpiLevel), and the kernels below decode its winners and count chain
// matches, each row against the chain of its own label (chain table, CSR over all nodes), per chain length L:
//   tor   = #{k : top1 == chain[k]}                                   -> hits_all          (main.py:158-160)
//   point = #{k : lvl[depth(chain[k])] == chain[k]}                   -> point             (main.py:182-189)
//   edge  = #{k < L-1 : match[k] and match[k+1]}  (L == 1: match[0])  -> edge / single-node path (main.py:179-185)
// hgr_hier_metrics_fused_rows runs both halves on one GPU; in the class-sharded form every rank runs the GEMM on its
// slice of the sorted bank and pushes its winners to the row owner (hier_push_kernel), which takes their max and
// finishes the rows (hier_finish_gathered_kernel) -- bit-identical to the one-GPU call.
//
// Tie rule = first position (what an arg-max over the masked array returns on the CPU): among equal values the
// smallest position j in `train_index` wins; a masked column holds exactly -1.0f, so when no in-level value exceeds -1
// the first position holding -1 wins -- `first_out[l]` is the first position whose column is NOT at level l.
#include "common.cuh"
#include "topk_list.cuh"

namespace hgr {
namespace {

constexpr int kMaxLevels = 32;   // levels of the per-level arg-max epilogue: one lane of a warp each in finish_row

__device__ __forceinline__ bool better(float v, int32_t j, float bv, int32_t bj) {
  return v > bv || (v == bv && j < bj);
}

// The per-level in-level maxima come from the GEMM epilogue as winner words (topk_list.cuh: order key << 32 | ~sorted
// bank row).  `finish_row` is run by one WARP per image row, lane = level (n_levels <= 32), so every load of a row is
// issued at once: it decodes the winners, maps the sorted bank row back to its position in `train_index`, and applies
// the rules above -- the -1 fill (first_out), first position among equal values, chain matching.  It returns the
// row's counts (warp-uniform).  L == 0 decodes the row and counts nothing.  `words(row, lane, n_levels)` gives the
// winner word of level lane (0: no column of that level): `WsWords` reads the one-GPU call's own workspace and hands it
// back zeroed; `GatheredWords` takes the max over the class shards' words in a peer-exchange slot.
// The caller passes L <= HGR_HIER_MAX_CHAIN = 32 = the lanes of a warp, so lane k takes chain entry k and the whole
// chain is matched in ONE ballot whatever L is: the warp votes sit under no branch on L (a per-row L from memory would
// otherwise make the compiler assume divergence there and spill).
static_assert(HGR_HIER_MAX_CHAIN <= 32, "finish_row matches a chain in one warp");

struct RowCounts {
  unsigned long long tor, point, edge;
};

// The one-GPU call's own workspace: read the word and hand it back zeroed, so the next call needs no memset.
struct WsWords {
  unsigned long long* __restrict__ lvl_best;
  __device__ __forceinline__ unsigned long long operator()(int64_t row, int lane, int n_levels) const {
    const unsigned long long w = lvl_best[row * n_levels + lane];
    lvl_best[row * n_levels + lane] = 0ull;
    return w;
  }
};

template <class Words>
__device__ __forceinline__ RowCounts finish_row(const Words& words, int64_t row, int lane, int64_t M, int n_levels,
                                                const int32_t* __restrict__ sorted_to_pos,
                                                const int32_t* __restrict__ first_out, const int32_t* __restrict__ chain,
                                                const int32_t* __restrict__ chain_level, int L,
                                                int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1) {
  float v = -INFINITY;          // in-level maximum of my level (before the -1 rule)
  int32_t j = 0x7FFFFFFF;       // its position in train_index
  int32_t node = 0;             // winner of my level after the -1 rule
  if (lane < n_levels) {
    const unsigned long long w = words(row, lane, n_levels);
    const int32_t fo = first_out[lane];
    if (w != 0ull) {
      v = winner_value(w);
      j = sorted_to_pos[winner_item(w)];
    }
    node = j;
    if (fo >= 0 && fo < M && better(-1.0f, fo, v, j)) node = fo;   // the masked array holds -1 at every out-of-level position
    if (node == 0x7FFFFFFF) node = 0;
    if (lvl_idx) lvl_idx[row * n_levels + lane] = node;
  }
  // overall top-1 over the train columns = best of the in-level maxima (value desc, position asc)
  float bv = v;
  int32_t bj = j;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int32_t oj = __shfl_xor_sync(0xffffffffu, bj, o);
    if (better(ov, oj, bv, bj)) {
      bv = ov;
      bj = oj;
    }
  }
  const int32_t t1 = bj == 0x7FFFFFFF ? -1 : bj;
  if (top1 && lane == 0) top1[row] = t1;
  // chain matching: lane k takes chain entry k; match[k] needs the winner of level chain_level[k]
  const int32_t p = lane < L ? chain[lane] : -2;
  const int cl = lane < L ? chain_level[lane] : -1;
  const int32_t win = __shfl_sync(0xffffffffu, node, cl >= 0 && cl < 32 ? cl : 0);
  const bool m = lane < L && cl >= 0 && cl < n_levels && win == p;
  const unsigned mm = __ballot_sync(0xffffffffu, m);
  RowCounts c;
  c.tor = __popc(__ballot_sync(0xffffffffu, lane < L && t1 == p));
  c.point = __popc(mm);
  c.edge = L == 1 ? c.point : __popc(mm & (mm << 1));   // match[k] and match[k - 1]
  return c;
}

// hgr_hier_metrics_fused_rows: every row is matched against the chain of its own label, looked up in the chain table
// (CSR over all nodes).  Counters are kept per chain length L ({rows, TOR hits, points, edges} in bin L), so they stay
// integer and exact; the reference's per-batch divisions by L - 1 and L follow on the host.  A block first reduces its
// rows into a shared histogram: in a single-label batch every row would otherwise hit the same four global words.
constexpr int kRowsPerBlock = 8;
constexpr int kHistWords = (HGR_HIER_MAX_CHAIN + 1) * 4;

// kSplits (node_splits != NULL): counter set s ([s][kHistWords]) takes the rows whose label has bit s in node_splits --
// a row in several splits is added to each of them.  Without splits there is one set and a 528-byte histogram.
template <bool kSplits, class Words>
__device__ __forceinline__ void finish_rows_block(const Words& words, int64_t B, int64_t M, int n_levels,
                                                  const int32_t* __restrict__ sorted_to_pos,
                                                  const int32_t* __restrict__ first_out,
                                                  const int32_t* __restrict__ targets, int64_t n_nodes,
                                                  const int32_t* __restrict__ chain_ptr,
                                                  const int32_t* __restrict__ chain_pos,
                                                  const int32_t* __restrict__ chain_level,
                                                  const uint8_t* __restrict__ node_splits, int n_sets,
                                                  int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1,
                                                  unsigned long long* counts) {
  constexpr int kSets = kSplits ? kMaxSplits : 1;
  __shared__ unsigned int s_cnt[kSets * kHistWords];   // <= kRowsPerBlock * HGR_HIER_MAX_CHAIN per word: 32 bits suffice
  for (int i = threadIdx.x; i < kSets * kHistWords; i += blockDim.x) s_cnt[i] = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kRowsPerBlock + (threadIdx.x >> 5);
  if (row < B) {                                            // warp-uniform
    // the row's chain; a target outside [0, n_nodes) or a chain length outside [1, HGR_HIER_MAX_CHAIN] is skipped
    // (decoded, so that lvl_idx / top1 are written and the workspace is zeroed, but counted nowhere)
    int32_t c0 = 0;
    int L = 0;
    if (lane == 0) {
      const int32_t t = targets[row];
      if (t >= 0 && t < n_nodes) {
        c0 = chain_ptr[t];
        L = chain_ptr[t + 1] - c0;
        if (L < 1 || L > HGR_HIER_MAX_CHAIN) L = 0;
      }
    }
    c0 = __shfl_sync(0xffffffffu, c0, 0);
    L = __shfl_sync(0xffffffffu, L, 0);
    const RowCounts c = finish_row(words, row, lane, M, n_levels, sorted_to_pos, first_out, chain_pos + c0,
                                   chain_level + c0, L, lvl_idx, top1);
    if (lane == 0 && L > 0) {
      const unsigned bits = kSplits ? node_splits[targets[row]] : 1u;   // L > 0: the target is a node
      for (int sp = 0; sp < kSets; ++sp) {
        if (!((bits >> sp) & 1u)) continue;
        unsigned int* bin = s_cnt + sp * kHistWords + 4 * L;
        atomicAdd(bin + 0, 1u);
        if (c.tor) atomicAdd(bin + 1, static_cast<unsigned int>(c.tor));
        if (c.point) atomicAdd(bin + 2, static_cast<unsigned int>(c.point));
        if (c.edge) atomicAdd(bin + 3, static_cast<unsigned int>(c.edge));
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < (kSplits ? n_sets : 1) * kHistWords; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(counts + i, static_cast<unsigned long long>(s_cnt[i]));
}

template <bool kSplits>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
hier_finish_rows_kernel(unsigned long long* __restrict__ lvl_best, int64_t B, int64_t M, int n_levels,
                        const int32_t* __restrict__ sorted_to_pos, const int32_t* __restrict__ first_out,
                        const int32_t* __restrict__ targets, int64_t n_nodes, const int32_t* __restrict__ chain_ptr,
                        const int32_t* __restrict__ chain_pos, const int32_t* __restrict__ chain_level,
                        const uint8_t* __restrict__ node_splits, int n_sets, int32_t* __restrict__ lvl_idx,
                        int32_t* __restrict__ top1, unsigned long long* counts) {
  finish_rows_block<kSplits>(WsWords{lvl_best}, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr,
                             chain_pos, chain_level, node_splits, n_sets, lvl_idx, top1, counts);
}

// ---- class-sharded form (hgr_hier_level_scatter / hgr_hier_finish_rows_gathered) -------------------------------------
// Every class shard runs the level GEMM on its contiguous slice [row_base, row_base + M_r) of the level-sorted train
// bank; hier_push_kernel rebases each winner word to the GLOBAL sorted row and stores it into region `rank` of the row
// owner's exchange slot ([n_parts][block_rows][n_levels] words).  The owner takes the max over its n_parts words per
// (row, level): that is the word the single-GPU epilogue's atomicMax would have left, because the word's order is
// (value desc, global sorted row asc), the level-sorted bank keeps train_index order inside a level, and max is
// associative.  The gathered words then go through the same finish_row.

// Max over the shards' words of a row; the exchange slot is read only (producers overwrite all of it every batch).
struct GatheredWords {
  const unsigned long long* __restrict__ parts;
  int n_parts;
  int64_t part_stride;
  __device__ __forceinline__ unsigned long long operator()(int64_t row, int lane, int n_levels) const {
    unsigned long long w = 0ull;
    for (int p = 0; p < n_parts; ++p) {
      const unsigned long long o = parts[p * part_stride + row * n_levels + lane];
      w = o > w ? o : w;
    }
    return w;
  }
};

template <bool kSplits>
__global__ void __launch_bounds__(kRowsPerBlock * 32)
hier_finish_gathered_kernel(const unsigned long long* __restrict__ parts, int n_parts, int64_t part_stride, int64_t B,
                            int64_t M, int n_levels, const int32_t* __restrict__ sorted_to_pos,
                            const int32_t* __restrict__ first_out, const int32_t* __restrict__ targets, int64_t n_nodes,
                            const int32_t* __restrict__ chain_ptr, const int32_t* __restrict__ chain_pos,
                            const int32_t* __restrict__ chain_level, const uint8_t* __restrict__ node_splits, int n_sets,
                            int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1, unsigned long long* counts) {
  finish_rows_block<kSplits>(GatheredWords{parts, n_parts, part_stride}, B, M, n_levels, sorted_to_pos, first_out,
                             targets, n_nodes, chain_ptr, chain_pos, chain_level, node_splits, n_sets, lvl_idx, top1,
                             counts);
}

struct HierDst {
  unsigned long long* p[kMaxScatterBlocks];
};

// One thread per (row, level) word of the shard's workspace: read it, hand it back zeroed, move its item from the
// shard's sorted row to the global one (0 = no column of that level here: stays 0) and store it -- zeros included, so
// a slot never holds anything of an earlier batch -- at its row owner.  Plain stores, local or peer memory; the
// hgr_peer_signal that follows in stream order publishes them.
constexpr int kPushThreads = 256;
__global__ void __launch_bounds__(kPushThreads)
hier_push_kernel(unsigned long long* __restrict__ lvl_best, int64_t n_words, int n_levels, int64_t block_rows,
                 uint32_t row_base, const __grid_constant__ HierDst dst) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kPushThreads + threadIdx.x;
  if (i >= n_words) return;
  unsigned long long w = lvl_best[i];
  lvl_best[i] = 0ull;
  if (w != 0ull) w = winner_word(static_cast<uint32_t>(w >> 32), static_cast<uint32_t>(winner_item(w)) + row_base);
  const int64_t row = i / n_levels;
  const int g = static_cast<int>(row / block_rows);
  dst.p[g][i - g * block_rows * n_levels] = w;
}

}  // namespace

int launch_hier_push(unsigned long long* lvl_best, int64_t B, int n_levels, int64_t row_base, int64_t block_rows,
                     int n_blocks, unsigned long long* const* dst, cudaStream_t stream) {
  HierDst d{};
  for (int g = 0; g < n_blocks; ++g) d.p[g] = dst[g];
  const int64_t n_words = B * n_levels;
  hier_push_kernel<<<static_cast<unsigned>((n_words + kPushThreads - 1) / kPushThreads), kPushThreads, 0, stream>>>(
      lvl_best, n_words, n_levels, block_rows, static_cast<uint32_t>(row_base), d);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_hier_finish_gathered(const unsigned long long* parts, int n_parts, int64_t part_stride, int64_t B, int64_t M,
                                int n_levels, const int32_t* sorted_to_pos, const int32_t* first_out,
                                const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                                const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits,
                                int n_sets, int32_t* lvl_idx, int32_t* top1, int64_t* counts, cudaStream_t stream) {
  const int blocks = static_cast<int>((B + kRowsPerBlock - 1) / kRowsPerBlock);     // one warp per image row
  auto kernel = node_splits ? hier_finish_gathered_kernel<true> : hier_finish_gathered_kernel<false>;
  kernel<<<blocks, kRowsPerBlock * 32, 0, stream>>>(parts, n_parts, part_stride, B, M, n_levels, sorted_to_pos, first_out,
                                                    targets, n_nodes, chain_ptr, chain_pos, chain_level, node_splits,
                                                    n_sets, lvl_idx, top1, reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_hier_finish_rows(unsigned long long* lvl_best, int64_t B, int64_t M, int n_levels, const int32_t* sorted_to_pos,
                            const int32_t* first_out, const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                            const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits, int n_sets,
                            int32_t* lvl_idx, int32_t* top1, int64_t* counts, cudaStream_t stream) {
  if (n_levels < 1 || n_levels > kMaxLevels)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics_fused_rows: %d levels outside [1, %d]", n_levels, kMaxLevels);
  const int blocks = static_cast<int>((B + kRowsPerBlock - 1) / kRowsPerBlock);     // one warp per image row
  auto kernel = node_splits ? hier_finish_rows_kernel<true> : hier_finish_rows_kernel<false>;
  kernel<<<blocks, kRowsPerBlock * 32, 0, stream>>>(lvl_best, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes,
                                                    chain_ptr, chain_pos, chain_level, node_splits, n_sets, lvl_idx, top1,
                                                    reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
