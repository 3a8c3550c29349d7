// TOR / POR hierarchical metrics of one single-label batch in ONE pass over the dense logits (SURVEY.md 8-f1).
//
// Reference: main.py:143,152-191.  Per batch the reference takes the arg-max over `train_index` (TOR, :155-160)
// and, for every node p of the label's ancestor chain, clones the [B, N] logits, fills every column that is not at
// p's depth with -1, gathers `train_index` and takes another arg-max (:163-176) -- L + 1 passes over B x N plus a
// Python B x L loop with device->host copies (:177-191).  Here one CTA per image row walks the train columns once,
// keeps a running (value, position) arg-max PER DEPTH LEVEL (the depth of a column is one int8 look-up), and then
// counts chain matches itself:
//   counts[0] += #{k : top1 == chain[k]}                                   -> hits_all          (main.py:158-160)
//   counts[1] += #{k : lvl[depth(chain[k])] == chain[k]}                   -> point             (main.py:182-189)
//   counts[2] += #{k < L-1 : match[k] and match[k+1]}  (L == 1: match[0])  -> edge / single-node path (main.py:179-185)
// HBM-bound: B * M * 4 bytes of logits read once (+ M * 5 bytes of column ids / levels from L2).
//
// Tie rule = first position (what an arg-max over the masked array returns on the CPU): among equal values the
// smallest position j in `cols` wins; a masked column holds exactly -1.0f, so when no in-level value exceeds -1 the
// first position holding -1 wins -- `first_out[l]` is the first position whose column is NOT at level l.
//
// The fused paths (hgr_hier_metrics_fused / _rows) apply the same rules to per-level winners taken in the GEMM
// epilogue; the _rows variant matches every row against the chain of its own label (batches that mix classes).
#include "common.cuh"
#include "topk_list.cuh"

namespace hgr {
namespace {

constexpr int kHierUnroll = 8;  // independent (column id -> level, logit) load chains in flight per thread
constexpr int kMaxLevels = 32;   // <= 16 levels: 256 threads per row; 17..32 levels: 128 threads (same 32 KB of slots)

struct Best {
  float v;
  int32_t j;
};
__device__ __forceinline__ bool better(float v, int32_t j, float bv, int32_t bj) {
  return v > bv || (v == bv && j < bj);
}

template <int kLevels, int kHierThreads>
__global__ void __launch_bounds__(kHierThreads)
hier_metrics_kernel(const float* __restrict__ logits, int64_t ldl, const int32_t* __restrict__ cols, int64_t M,
                    const int8_t* __restrict__ level, int n_levels, const int32_t* __restrict__ first_out,
                    const int32_t* __restrict__ chain, const int32_t* __restrict__ chain_level, int L,
                    int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1, unsigned long long* counts) {
  __shared__ float s_v[kLevels][kHierThreads];
  __shared__ int32_t s_j[kLevels][kHierThreads];
  __shared__ float s_wv[kLevels][kHierThreads / 32];
  __shared__ int32_t s_wj[kLevels][kHierThreads / 32];
  __shared__ int32_t s_node[kLevels];      // winner node per level (after the -1 rule)
  __shared__ float s_tv[kLevels];          // in-level maxima (before the -1 rule): their best is the TOR top-1
  __shared__ int32_t s_tj[kLevels];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t row = blockIdx.x;
  const float* lr = logits + row * ldl;
  for (int l = 0; l < n_levels; ++l) {
    s_v[l][tid] = -INFINITY;
    s_j[l][tid] = 0x7FFFFFFF;
  }
  // one pass: positions tid, tid + 128, ... (ascending per thread, so `>` keeps the first of equal values)
  for (int64_t j0 = tid; j0 < M; j0 += kHierUnroll * kHierThreads) {
    int32_t c[kHierUnroll];
    int l[kHierUnroll];
    float v[kHierUnroll];
#pragma unroll
    for (int u = 0; u < kHierUnroll; ++u) {
      const int64_t j = j0 + u * kHierThreads;
      c[u] = j < M ? (cols ? __ldg(cols + j) : static_cast<int32_t>(j)) : -1;
    }
#pragma unroll
    for (int u = 0; u < kHierUnroll; ++u) {
      l[u] = c[u] >= 0 ? __ldg(level + c[u]) : -1;
      v[u] = c[u] >= 0 ? __ldg(lr + c[u]) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kHierUnroll; ++u) {
      if (l[u] >= 0 && l[u] < n_levels && v[u] > s_v[l[u]][tid]) {
        s_v[l[u]][tid] = v[u];
        s_j[l[u]][tid] = static_cast<int32_t>(j0 + u * kHierThreads);
      }
    }
  }
  // per level: block arg-max by (value desc, position asc)
  for (int l = 0; l < n_levels; ++l) {
    float v = s_v[l][tid];
    int32_t j = s_j[l][tid];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, v, o);
      const int32_t oj = __shfl_xor_sync(0xffffffffu, j, o);
      if (better(ov, oj, v, j)) {
        v = ov;
        j = oj;
      }
    }
    if (lane == 0) {
      s_wv[l][warp] = v;
      s_wj[l][warp] = j;
    }
  }
  __syncthreads();
  if (tid <= n_levels) {
    if (tid < n_levels) {
      float v = s_wv[tid][0];
      int32_t j = s_wj[tid][0];
      for (int w = 1; w < kHierThreads / 32; ++w)
        if (better(s_wv[tid][w], s_wj[tid][w], v, j)) {
          v = s_wv[tid][w];
          j = s_wj[tid][w];
        }
      s_tv[tid] = v;
      s_tj[tid] = j;
      // the masked array holds -1 at every out-of-level position (main.py:171)
      const int32_t fo = first_out[tid];
      if (fo >= 0 && fo < M && better(-1.0f, fo, v, j)) {
        v = -1.0f;
        j = fo;
      }
      if (j == 0x7FFFFFFF) j = 0;  // M == 0 cannot happen (checked on the host); defensive
      const int32_t node = cols ? cols[j] : j;
      s_node[tid] = node;
      if (lvl_idx) lvl_idx[row * n_levels + tid] = node;
    }
  }
  __syncthreads();
  if (tid == 0) {
    // overall top-1 over the train columns (main.py:155-156) = best of the per-level in-level maxima
    float bv = -INFINITY;
    int32_t bj = 0x7FFFFFFF;
    for (int l = 0; l < n_levels; ++l)
      if (s_tj[l] != 0x7FFFFFFF && better(s_tv[l], s_tj[l], bv, bj)) {
        bv = s_tv[l];
        bj = s_tj[l];
      }
    const int32_t t1 = bj == 0x7FFFFFFF ? -1 : (cols ? cols[bj] : bj);
    if (top1) top1[row] = t1;
    unsigned long long tor = 0, point = 0, edge = 0;
    bool prev = false;
    for (int k = 0; k < L; ++k) {
      const int32_t p = chain[k];
      tor += (t1 == p);
      const int cl = chain_level[k];
      const bool m = cl >= 0 && cl < n_levels && s_node[cl] == p;
      point += m;
      if (k > 0) edge += (prev && m);
      prev = m;
    }
    if (L == 1) edge = prev ? 1 : 0;
    if (tor) atomicAdd(counts + 0, tor);
    if (point) atomicAdd(counts + 1, point);
    if (edge) atomicAdd(counts + 2, edge);
  }
}

// Second half of the FUSED paths: the per-level in-level maxima come from the GEMM epilogue (score_pair.cu, kEpiLevel)
// as winner words (topk_list.cuh: order key << 32 | ~sorted bank row).  `finish_row` is run by one WARP per image row,
// lane = level (n_levels <= 32), so every load of a row is issued at once: it decodes the winners, maps the sorted bank
// row back to its position in `train_index`, and applies the same rules as the kernel above -- the -1 fill (first_out),
// first position among equal values, chain matching.  It returns the row's counts (warp-uniform).  L == 0 decodes the
// row and counts nothing.  `words(row, lane, n_levels)` gives the winner word of level lane (0: no column of that
// level): `WsWords` reads the fused call's own workspace and hands it back zeroed; `GatheredWords` takes the max over
// the class shards' words in a peer-exchange slot.
// kMaxChain: the longest chain the caller passes (<= 64).  At 32 the chain is matched in ONE group of 32 whatever L is,
// so the warp votes sit under no branch on L (a per-row L from memory would otherwise make the compiler assume
// divergence there and spill).
struct RowCounts {
  unsigned long long tor, point, edge;
};

// The fused calls' own workspace: read the word and hand it back zeroed, so the next call needs no memset.
struct WsWords {
  unsigned long long* __restrict__ lvl_best;
  __device__ __forceinline__ unsigned long long operator()(int64_t row, int lane, int n_levels) const {
    const unsigned long long w = lvl_best[row * n_levels + lane];
    lvl_best[row * n_levels + lane] = 0ull;
    return w;
  }
};

template <int kMaxChain, class Words>
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
  // chain matching: lane k takes chain entries k, k + 32 (L <= 64); match[k] needs the winner of level chain_level[k]
  RowCounts c{0, 0, 0};
  bool carry = false;           // match[k0 - 1] of the previous group of 32
  const int k_end = kMaxChain <= 32 ? 32 : L;
  for (int k0 = 0; k0 < k_end; k0 += 32) {
    const int k = k0 + lane;
    const int32_t p = k < L ? chain[k] : -2;
    const int cl = k < L ? chain_level[k] : -1;
    const int32_t win = __shfl_sync(0xffffffffu, node, cl >= 0 && cl < 32 ? cl : 0);
    const bool m = k < L && cl >= 0 && cl < n_levels && win == p;
    const unsigned mm = __ballot_sync(0xffffffffu, m);
    c.tor += __popc(__ballot_sync(0xffffffffu, k < L && t1 == p));
    c.point += __popc(mm);
    c.edge += __popc(mm & ((mm << 1) | (carry ? 1u : 0u)));   // match[k] and match[k - 1]
    carry = (mm >> 31) & 1u;
  }
  if (L == 1) c.edge = c.point;
  return c;
}

// hgr_hier_metrics_fused: one chain for the whole batch, three counters.
__global__ void __launch_bounds__(128)
hier_finish_kernel(unsigned long long* __restrict__ lvl_best, int64_t B, int64_t M, int n_levels,
                   const int32_t* __restrict__ sorted_to_pos, const int32_t* __restrict__ first_out,
                   const int32_t* __restrict__ chain, const int32_t* __restrict__ chain_level, int L,
                   int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1, unsigned long long* counts) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= B) return;
  const RowCounts c = finish_row<64>(WsWords{lvl_best}, row, lane, M, n_levels, sorted_to_pos,
                                     first_out, chain, chain_level, L, lvl_idx, top1);
  if (lane == 0) {
    if (c.tor) atomicAdd(counts + 0, c.tor);
    if (c.point) atomicAdd(counts + 1, c.point);
    if (c.edge) atomicAdd(counts + 2, c.edge);
  }
}

// hgr_hier_metrics_fused_rows: every row is matched against the chain of its own label, looked up in the chain table
// (CSR over all nodes).  Counters are kept per chain length L ({rows, TOR hits, points, edges} in bin L), so they stay
// integer and exact; the reference's per-batch divisions by L - 1 and L follow on the host.  A block first reduces its
// rows into a shared histogram: in a single-label batch every row would otherwise hit the same four global words.
constexpr int kRowsPerBlock = 8;
constexpr int kHistWords = (HGR_HIER_MAX_CHAIN + 1) * 4;

template <class Words>
__device__ __forceinline__ void finish_rows_block(const Words& words, int64_t B, int64_t M, int n_levels,
                                                  const int32_t* __restrict__ sorted_to_pos,
                                                  const int32_t* __restrict__ first_out,
                                                  const int32_t* __restrict__ targets, int64_t n_nodes,
                                                  const int32_t* __restrict__ chain_ptr,
                                                  const int32_t* __restrict__ chain_pos,
                                                  const int32_t* __restrict__ chain_level, int32_t* __restrict__ lvl_idx,
                                                  int32_t* __restrict__ top1, unsigned long long* counts) {
  __shared__ unsigned int s_cnt[kHistWords];      // <= kRowsPerBlock * HGR_HIER_MAX_CHAIN per word: 32 bits suffice
  for (int i = threadIdx.x; i < kHistWords; i += blockDim.x) s_cnt[i] = 0u;
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
    const RowCounts c = finish_row<HGR_HIER_MAX_CHAIN>(words, row, lane, M, n_levels, sorted_to_pos,
                                                       first_out, chain_pos + c0, chain_level + c0, L, lvl_idx, top1);
    if (lane == 0 && L > 0) {
      unsigned int* bin = s_cnt + 4 * L;
      atomicAdd(bin + 0, 1u);
      if (c.tor) atomicAdd(bin + 1, static_cast<unsigned int>(c.tor));
      if (c.point) atomicAdd(bin + 2, static_cast<unsigned int>(c.point));
      if (c.edge) atomicAdd(bin + 3, static_cast<unsigned int>(c.edge));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kHistWords; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(counts + i, static_cast<unsigned long long>(s_cnt[i]));
}

__global__ void __launch_bounds__(kRowsPerBlock * 32)
hier_finish_rows_kernel(unsigned long long* __restrict__ lvl_best, int64_t B, int64_t M, int n_levels,
                        const int32_t* __restrict__ sorted_to_pos, const int32_t* __restrict__ first_out,
                        const int32_t* __restrict__ targets, int64_t n_nodes, const int32_t* __restrict__ chain_ptr,
                        const int32_t* __restrict__ chain_pos, const int32_t* __restrict__ chain_level,
                        int32_t* __restrict__ lvl_idx, int32_t* __restrict__ top1, unsigned long long* counts) {
  finish_rows_block(WsWords{lvl_best}, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr, chain_pos,
                    chain_level, lvl_idx, top1, counts);
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

__global__ void __launch_bounds__(kRowsPerBlock * 32)
hier_finish_gathered_kernel(const unsigned long long* __restrict__ parts, int n_parts, int64_t part_stride, int64_t B,
                            int64_t M, int n_levels, const int32_t* __restrict__ sorted_to_pos,
                            const int32_t* __restrict__ first_out, const int32_t* __restrict__ targets, int64_t n_nodes,
                            const int32_t* __restrict__ chain_ptr, const int32_t* __restrict__ chain_pos,
                            const int32_t* __restrict__ chain_level, int32_t* __restrict__ lvl_idx,
                            int32_t* __restrict__ top1, unsigned long long* counts) {
  finish_rows_block(GatheredWords{parts, n_parts, part_stride}, B, M, n_levels, sorted_to_pos, first_out, targets,
                    n_nodes, chain_ptr, chain_pos, chain_level, lvl_idx, top1, counts);
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
                                const int32_t* chain_pos, const int32_t* chain_level, int32_t* lvl_idx, int32_t* top1,
                                int64_t* counts, cudaStream_t stream) {
  const int blocks = static_cast<int>((B + kRowsPerBlock - 1) / kRowsPerBlock);     // one warp per image row
  hier_finish_gathered_kernel<<<blocks, kRowsPerBlock * 32, 0, stream>>>(
      parts, n_parts, part_stride, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr, chain_pos,
      chain_level, lvl_idx, top1, reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_hier_finish(unsigned long long* lvl_best, int64_t B, int64_t M, int n_levels, const int32_t* sorted_to_pos,
                       const int32_t* first_out, const int32_t* chain, const int32_t* chain_level, int L, int32_t* lvl_idx,
                       int32_t* top1, int64_t* counts, cudaStream_t stream) {
  if (n_levels < 1 || n_levels > kMaxLevels)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics_fused: %d levels outside [1, %d]", n_levels, kMaxLevels);
  const int blocks = static_cast<int>((B + 3) / 4);     // one warp per image row
  hier_finish_kernel<<<blocks, 128, 0, stream>>>(lvl_best, B, M, n_levels, sorted_to_pos, first_out, chain, chain_level, L,
                                                 lvl_idx, top1, reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_hier_finish_rows(unsigned long long* lvl_best, int64_t B, int64_t M, int n_levels, const int32_t* sorted_to_pos,
                            const int32_t* first_out, const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                            const int32_t* chain_pos, const int32_t* chain_level, int32_t* lvl_idx, int32_t* top1,
                            int64_t* counts, cudaStream_t stream) {
  if (n_levels < 1 || n_levels > kMaxLevels)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics_fused_rows: %d levels outside [1, %d]", n_levels, kMaxLevels);
  const int blocks = static_cast<int>((B + kRowsPerBlock - 1) / kRowsPerBlock);     // one warp per image row
  hier_finish_rows_kernel<<<blocks, kRowsPerBlock * 32, 0, stream>>>(
      lvl_best, B, M, n_levels, sorted_to_pos, first_out, targets, n_nodes, chain_ptr, chain_pos, chain_level, lvl_idx,
      top1, reinterpret_cast<unsigned long long*>(counts));
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_hier_metrics(const float* logits, int64_t ldl, int64_t B, const int32_t* cols, int64_t M,
                        const int8_t* level, int n_levels, const int32_t* first_out, const int32_t* chain,
                        const int32_t* chain_level, int L, int32_t* lvl_idx, int32_t* top1, int64_t* counts,
                        cudaStream_t stream) {
  if (n_levels < 1 || n_levels > kMaxLevels)
    return set_error(HGR_ERR_UNSUPPORTED, "hgr_hier_metrics: %d levels outside [1, %d]", n_levels, kMaxLevels);
  unsigned long long* cnt = reinterpret_cast<unsigned long long*>(counts);
  if (n_levels <= 16)
    hier_metrics_kernel<16, 256><<<static_cast<unsigned>(B), 256, 0, stream>>>(
        logits, ldl, cols, M, level, n_levels, first_out, chain, chain_level, L, lvl_idx, top1, cnt);
  else
    hier_metrics_kernel<32, 128><<<static_cast<unsigned>(B), 128, 0, stream>>>(
        logits, ldl, cols, M, level, n_levels, first_out, chain, chain_level, L, lvl_idx, top1, cnt);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
