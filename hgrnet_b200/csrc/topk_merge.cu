// Merge the partial top-K lists of one image row into the final sorted top-K, map bank rows to
// node ids and count Hit@{1,2,5,10,20}.
//
// Reference: the tail of the eval reductions in main.test -- `model.test_index[pred]`,
// `pred.eq(targets)`, `correct[:k].sum()` (main.py:139-147) -- and, for the class-sharded
// multi-GPU head, the combination of the per-rank lists after the NCCL all-gather.
//
// One warp per row, kMergeWarps rows per CTA.  The CTA first stages all lists of its rows in
// shared memory (coalesced), then each warp runs K rounds of a P-way merge (merge_heads): lane l owns lists
// l, l+32, ...; per round the lane-local best head, a warp arg-max by (value desc, list asc),
// and the winner advances its head (shared-memory read).  Heads compare by (value desc, item
// asc), every list is itself sorted that way, so the result is ordered (value desc, bank row asc)
// -- deterministic whatever way the producers interleave bank rows over lists.
//
// Speculative lists (KL < K, tcgen05 path): the row is CERTIFIED when every full list ends strictly
// below the merged K-th value (narrow_tails) -- anything such a list dropped is <= its last entry, hence
// cannot belong to (or tie with) the top-K.  An uncertified row is re-scanned exactly by its warp on the
// CUDA cores (repair_lists, simt_row.cuh).  With randomly ordered bank rows this is a ~1e-8-per-row event.
#include "common.cuh"
#include "placement.cuh"
#include "simt_row.cuh"

namespace hgr {
namespace {

constexpr int kMergeWarps = 4;

constexpr int kDoubtWords = 10;  // bit per list, up to 320 lists per row

// Rank `lane` of a list replicated in every lane.
__device__ __forceinline__ Cand lane_entry(const SortedList<HGR_TOPK_MAX>& list, int lane) {
  Cand c;
  c.v = -INFINITY;
  c.i = -1;
#pragma unroll
  for (int k = 0; k < HGR_TOPK_MAX; ++k) {
    if (lane == k) {
      c.v = list.v[k];
      c.i = list.i[k];
    }
  }
  return c;
}

// Offers the valid entries (item >= 0) of a list of n to `full`, in list order.
__device__ __forceinline__ void insert_entries(SortedList<HGR_TOPK_MAX>& full, const float* val, const int32_t* idx, int n) {
  for (int k = 0; k < n; ++k) {
    const int32_t it = idx[k];
    const float v = val[k];
    if (it >= 0 && v > full.thr()) full.insert(v, it);
  }
}

// The two exact repairs below (repair_lists, repair_shards) are written once and fill a replicated list `full`.  The
// kernels reach them only through the cold __noinline__ repair_cold of their argument type, so that everything the
// rare repair needs (two 32-entry lists) lives outside the merge kernels, which keep their register count.  repair_cold
// takes a pointer to the kernel's __grid_constant__ parameter (handed over by value, the whole argument block would be
// copied to the stack of every thread at kernel entry) and returns rank `lane` of the repaired row.

// ---- exact repair of the scoring kernel's own lists (repair_lists) ----------------------------------------------
// A row -- or split s of a row -- whose speculative lists could not all be certified.  Only the column ranges of the
// DOUBTFUL lists (bits of `dmask`) are re-scanned on the CUDA cores (1 / lists-per-row of the bank each); the entries of
// the certified lists are final as they are (whatever such a list dropped is below the old K-th value, which can only
// rise) and are inserted as candidates.  Slots are visited in ascending column order and SortedList keeps the first of
// equal values, so the result has the documented (value desc, bank row asc) order.
// slot_cols: bank rows [c0, c1) of list slot p of row tile mt, and whether the slot takes part in split s.
//  * MergeArgs: slot p is worker first_cta(mt) + p, its chunk of flattened units clipped to the tile; every slot counts.
//  * SplitMergeArgs: slot p of the grouped schedule (group_slot_range); it counts when its group is in split s.
__device__ __forceinline__ bool slot_cols(const MergeArgs& a, int32_t mt, int p, int, int64_t& c0, int64_t& c1) {
  const int64_t t0 = static_cast<int64_t>(mt) * a.sched.U;
  const int32_t w = a.sched.first_cta(mt) + p;
  int64_t u0 = a.sched.unit_begin(w) - t0, u1 = a.sched.unit_begin(w + 1) - t0;
  u0 = u0 < 0 ? 0 : u0;
  u1 = u1 > a.sched.U ? a.sched.U : u1;
  c0 = u0 * kUnit;
  c1 = u1 * kUnit;
  c1 = c1 > a.C ? a.C : c1;
  return true;
}
__device__ __forceinline__ bool slot_cols(const SplitMergeArgs& a, int32_t mt, int p, int s, int64_t& c0, int64_t& c1) {
  const int g = group_slot_range(a.sched, a.groups, mt, p, c0, c1);
  return (a.group_splits[g] >> s) & 1u;
}
__device__ __forceinline__ int64_t list_stride(const MergeArgs& a) { return a.part_stride > 0 ? a.part_stride : a.B * a.KL; }
__device__ __forceinline__ int64_t list_stride(const SplitMergeArgs& a) { return a.B * a.KL; }

template <class Args>
__device__ __forceinline__ void repair_lists(const Args* a, int64_t row, int lane, int cnt, int s, const uint32_t* dmask,
                                             SortedList<HGR_TOPK_MAX>& full) {
  const int KL = a->KL;
  const int64_t pstride = list_stride(*a);
  const int32_t mt = static_cast<int32_t>(row / a->sched.rows);
  for (int p = 0; p < cnt; ++p) {
    int64_t c0, c1;
    if (!slot_cols(*a, mt, p, s, c0, c1)) continue;
    if ((dmask[p >> 5] >> (p & 31)) & 1u)
      scan_row_range_lanes<HGR_TOPK_MAX>(reinterpret_cast<const uint4*>(a->X) + row * a->D8,
                                         reinterpret_cast<const uint4*>(a->bank), c0, c1, a->D8, lane, full);
    else
      insert_entries(full, a->part_val + p * pstride + row * KL, a->part_idx + p * pstride + row * KL, KL);
  }
}

// ---- exact repair from the shard table (repair_shards) ----------------------------------------------------------
// Owner side of the class-sharded head: list p of a row is class shard p's final local top-K (node ids, values scaled
// by the producer).  A doubtful shard (bit p of `dm`: its bound reaches the merged K-th value) is re-scanned completely
// with the row's features -- over NVLink when the bank is a peer's --, its exact local top-K mapped to node ids and
// scaled like the producer did; the lists of the other shards are final as they are (what such a shard dropped is
// below the old K-th value, which can only rise).  Shards are visited in ascending order and SortedList keeps the first
// of equal values, so the tie order stays (value desc, shard asc, local row asc).  All HGR_TOPK_MAX entries of a
// re-scanned shard are offered (an unrolled loop keeps its list in registers), but only ranks < K of the result are
// kept, and those are the same as with K entries: the shard's entry of rank k >= K sorts behind K entries of its own
// shard (values >= its own -- the scale keeps the order -- offered earlier), so it can only land at rank K or later.
//  * MergeArgs (hgr_topk_merge_certified): every row of a shard; list p at p * part_stride + row * K.
//  * SplitCertArgs (hgr_topk_merge_splits_certified), split s: the shard rows whose node has bit s in node_splits;
//    list p at s * split_stride + p * part_stride + row * K.
struct SplitRows {   // bank rows of a shard whose node is in split s
  static constexpr bool kFilter = true;
  const int32_t* col_id;
  int32_t id_base;
  const uint8_t* node_splits;
  int64_t n_nodes;
  int s;
  __device__ __forceinline__ bool operator()(int64_t c) const {
    const int64_t node = col_id ? col_id[c] : id_base + c;
    return node >= 0 && node < n_nodes && ((node_splits[node] >> s) & 1u);
  }
};
__device__ __forceinline__ EveryRow shard_rows(const MergeArgs&, const hgr_shard_t&, int) { return EveryRow(); }
__device__ __forceinline__ SplitRows shard_rows(const SplitCertArgs& a, const hgr_shard_t& sh, int s) {
  return SplitRows{sh.col_id, sh.id_base, a.node_splits, a.n_nodes, s};
}
__device__ __forceinline__ int64_t shard_list(const MergeArgs& a, int p, int64_t row, int) {
  return p * (a.part_stride > 0 ? a.part_stride : a.B * a.K) + row * a.K;
}
__device__ __forceinline__ int64_t shard_list(const SplitCertArgs& a, int p, int64_t row, int s) {
  return s * a.split_stride + p * a.part_stride + row * a.K;
}
__device__ __forceinline__ float shard_scale(const MergeArgs& a) { return a.shard_scale; }
__device__ __forceinline__ float shard_scale(const SplitCertArgs& a) { return a.scale; }

template <class Args>
__device__ __forceinline__ void repair_shards(const Args* a, int64_t row, int lane, int s, unsigned dm,
                                              SortedList<HGR_TOPK_MAX>& full) {
  const int K = a->K;
  const uint4* xr = reinterpret_cast<const uint4*>(a->xrows) + row * a->xD8;
  for (int p = 0; p < static_cast<int>(a->P); ++p) {
    if ((dm >> p) & 1u) {
      const hgr_shard_t sh = a->shards[p];
      SortedList<HGR_TOPK_MAX> sub;
      sub.init();
      scan_row_range_lanes<HGR_TOPK_MAX>(xr, reinterpret_cast<const uint4*>(sh.bank), 0, sh.C, a->xD8, lane, sub,
                                         shard_rows(*a, sh, s));
#pragma unroll
      for (int k = 0; k < HGR_TOPK_MAX; ++k) {
        const int32_t it = sub.i[k];
        const float v = sub.v[k] * shard_scale(*a);
        if (it >= 0 && v > full.thr()) full.insert(v, sh.col_id ? sh.col_id[it] : sh.id_base + it);
      }
    } else {
      const int64_t l = shard_list(*a, p, row, s);
      insert_entries(full, a->part_val + l, a->part_idx + l, K);
    }
  }
}

// MergeArgs (one call site for both repairs): from the shard table when the global certificate failed (dm_global != 0),
// else of the row's own speculative lists.  The list lives in repair_cold's frame and the repairs run in functions of
// their own: under the 72-register budget of these kernels a list held in registers would spill.
__device__ __noinline__ void repair_row(const MergeArgs* a, int64_t row, int lane, int cnt, const uint32_t* dmask,
                                        SortedList<HGR_TOPK_MAX>& full) {
  repair_lists(a, row, lane, cnt, 0, dmask, full);
}
__device__ __noinline__ void repair_row_global(const MergeArgs* a, int64_t row, int lane, unsigned dm,
                                               SortedList<HGR_TOPK_MAX>& full) {
  repair_shards(a, row, lane, 0, dm, full);
}
__device__ __noinline__ Cand repair_cold(const MergeArgs* a, int64_t row, int lane, int cnt, const uint32_t* dmask,
                                         unsigned dm_global) {
  SortedList<HGR_TOPK_MAX> full;
  full.init();
  if (dm_global != 0u) {
    if (lane == 0 && a->repair_count) atomicAdd(a->repair_count, 1u);
    repair_row_global(a, row, lane, dm_global, full);
  } else {
    if (lane == 0 && a->rescan_count) atomicAdd(a->rescan_count, 1u);
    repair_row(a, row, lane, cnt, dmask, full);
  }
  return lane_entry(full, lane);
}
// SplitMergeArgs (split s of a row) and SplitCertArgs (split s of an owned row of the class-sharded head).
__device__ __noinline__ Cand repair_cold(const SplitMergeArgs* a, int64_t row, int lane, int cnt, int s,
                                         const uint32_t* dmask) {
  SortedList<HGR_TOPK_MAX> full;
  full.init();
  if (lane == 0 && a->rescan_count) atomicAdd(a->rescan_count, 1u);
  repair_lists(a, row, lane, cnt, s, dmask, full);
  return lane_entry(full, lane);
}
__device__ __noinline__ Cand repair_cold(const SplitCertArgs* a, int64_t row, int lane, int s, unsigned dm) {
  if (lane == 0 && a->repair_count) atomicAdd(a->repair_count, 1u);
  SortedList<HGR_TOPK_MAX> full;
  full.init();
  repair_shards(a, row, lane, s, dm, full);
  return lane_entry(full, lane);
}

// Lists of a row: P, or -- for the scoring kernel's own lists -- one per worker of the row's tile.
__device__ __forceinline__ int row_lists(const MergeArgs& a, int64_t row) {
  return a.use_sched ? a.sched.parts(static_cast<int32_t>(row / a.sched.rows)) : static_cast<int>(a.P);
}

// Hit@k counters of the block's rows (s_hits) into the global ones, one atomic per cut-off.  `tid` = threadIdx.x, read
// by the kernel, where it keeps the range its launch bounds give it (read in here, it loses it: more spills).
__device__ __forceinline__ void flush_hits(const MergeArgs& a, const int* s_hits, int tid) {
  __syncthreads();
  if (a.hits && tid < HGR_NUM_HITS && s_hits[tid] != 0)
    atomicAdd(reinterpret_cast<unsigned long long*>(a.hits) + tid, static_cast<unsigned long long>(s_hits[tid]));
}

// The ksel <= 32 winners of a row, compacted into win[0, ksel) as winner words in any order: lane r < ksel gets rank r
// (ranked by counting -- the words are distinct).
__device__ __forceinline__ void rank_winners(unsigned long long* win, int ksel, int lane, float& my_v, int32_t& my_i) {
  __syncwarp();
  unsigned long long mine = 0;
  int rank = 0;
  if (lane < ksel) {
    mine = win[lane];
    for (int j = 0; j < ksel; ++j) rank += win[j] > mine;
  }
  __syncwarp();
  if (lane < ksel) win[rank] = mine;
  __syncwarp();
  if (lane < ksel) {
    my_v = winner_value(win[lane]);
    my_i = winner_item(win[lane]);
  }
}

// Tail shared by both merge kernels.  Lane r holds rank r of the merged list (my_v, my_i = bank row or -1).
// `dmask` (per-warp shared memory, one bit per list): full speculative lists that end at or above the merged K-th
// value -> the row is repaired exactly (repair_cold).  Then: bank row -> node id, scale, store (dense or row-block
// scatter), Hit@k.
// `tailmax`: lane-local largest last entry of a FULL narrow list (-inf: none; narrow_tails) -- what the producer of a
// class shard reports as its bound when the certificate is left to the owner of the row (scatter.emit_bound).
__device__ __forceinline__ void finish_row(const MergeArgs& a, int64_t row, int lane, float my_v, int32_t my_i,
                                           bool doubt, const uint32_t* dmask, int cnt, int* s_hits,
                                           float tailmax = -INFINITY) {
  const int K = a.K;
  const bool emit_bound = a.scatter.n_blocks > 0 && a.scatter.emit_bound != 0;
  unsigned dm = 0u;
  if (a.part_bound != nullptr) {  // owner side of the global certificate: list p = shard p
    const float kth = __shfl_sync(0xffffffffu, my_i >= 0 ? my_v : -INFINITY, K - 1);
    const float bnd = lane < a.P ? a.part_bound[lane * a.bound_stride + row] : -INFINITY;
    dm = __ballot_sync(0xffffffffu, bnd > -INFINITY && bnd >= kth);
  }
  const bool local_doubt = a.KL < K && !emit_bound && __any_sync(0xffffffffu, doubt);
  if (dm != 0u || local_doubt) {
    __syncwarp();
    const Cand c = repair_cold(&a, row, lane, cnt, dmask, dm);
    my_v = c.v;
    my_i = c.i;
  }
  int32_t gid = -1;
  if (lane < K && my_i >= 0) gid = a.col_id ? a.col_id[my_i] : a.id_base + my_i;
  if (lane < K) {
    float* ov = a.topk_val;
    int32_t* oi = a.topk_idx;
    int64_t orow = row;
    if (a.scatter.n_blocks > 0) {  // row-block scatter (possibly into peer memory)
      const int64_t g = row / a.scatter.block_rows;
      ov = a.scatter.val[g];
      oi = a.scatter.idx[g];
      orow = row - g * a.scatter.block_rows;
    }
    ov[orow * K + lane] = my_i >= 0 ? my_v * a.scale : -INFINITY;
    oi[orow * K + lane] = gid;
  }
  if (emit_bound) {
    const float b = warp_max_f32(a.KL < K ? tailmax : -INFINITY);   // K-entry lists drop nothing that could matter
    if (lane == 0) {
      const int64_t g = row / a.scatter.block_rows;
      a.scatter.bound[g][row - g * a.scatter.block_rows] = b * a.scale;
    }
  }
  if (a.hits && a.targets) {
    const int32_t target = a.targets[row];
    const unsigned m = __ballot_sync(0xffffffffu, lane < K && gid >= 0 && gid == target);
    if (lane == 0 && m != 0 && target >= 0) {
      const int pos = __ffs(m) - 1;
#pragma unroll
      for (int c = 0; c < HGR_NUM_HITS; ++c)
        if (pos < hit_cut(c)) atomicAdd(&s_hits[c], 1);
    }
  }
}

// ---- K rounds of the P-way merge of sorted lists in shared memory (merge_heads) ---------------------------------
// lv / li: the warp's lists, [list][KL], each sorted (value desc, item asc).  Lane l owns lists l, l + 32, ...; live[q]
// says whether list lane + 32 q takes part.  Per round the lane-local best head, a warp arg-max by (value desc, item
// asc), and the lowest lane holding the winner advances that list.  Lane r gets rank r of the result in (my_v, my_i),
// (-inf, -1) past the last candidate.  Returns the K-th value (-inf: fewer than K candidates).
template <int kMaxListsPerLane>
__device__ __forceinline__ float merge_heads(const float* lv, const int32_t* li, int KL, int K,
                                             const bool (&live)[kMaxListsPerLane], int lane, float& my_v, int32_t& my_i) {
  int head[kMaxListsPerLane];
  float hv[kMaxListsPerLane];   // value of the current head of my q-th list (-inf: exhausted)
  int32_t hi[kMaxListsPerLane]; // its item (bank row / node id)
#pragma unroll
  for (int q = 0; q < kMaxListsPerLane; ++q) {
    const int p = lane + 32 * q;
    head[q] = 0;
    hi[q] = live[q] ? li[p * KL] : -1;
    hv[q] = hi[q] >= 0 ? lv[p * KL] : -INFINITY;
  }
  my_v = -INFINITY;
  my_i = -1;
  float kth = -INFINITY;
  for (int r = 0; r < K; ++r) {
    // lane-local best head, then warp arg-max; order: value desc, item asc
    float bv = hv[0];
    int32_t bi = hi[0];
#pragma unroll
    for (int q = 1; q < kMaxListsPerLane; ++q) {
      if (hv[q] > bv || (hv[q] == bv && hi[q] < bi && hi[q] >= 0)) {
        bv = hv[q];
        bi = hi[q];
      }
    }
    const float lbv = bv;
    const int32_t lbi = bi;
    // warp arg-max with two REDUX instructions: max of an order-preserving integer image of the value, then
    // the smallest item among the lanes that hold that value
    const uint32_t lkey = order_key(lbv);
    const uint32_t mkey = __reduce_max_sync(0xffffffffu, lkey);
    const uint32_t mitem =
        __reduce_min_sync(0xffffffffu, (lkey == mkey && lbi >= 0) ? static_cast<uint32_t>(lbi) : 0xFFFFFFFFu);
    if (mitem == 0xFFFFFFFFu) {  // every list exhausted: fewer than K candidates, the rest stays (-inf, -1)
      kth = -INFINITY;
      break;
    }
    bv = order_key_value(mkey);
    bi = static_cast<int32_t>(mitem);
    kth = bv;
    // the lowest lane holding the winner advances that list
    const unsigned holders = __ballot_sync(0xffffffffu, lbv == bv && lbi == bi);
    if (lane == __ffs(holders) - 1) {
      bool done = false;
#pragma unroll
      for (int q = 0; q < kMaxListsPerLane; ++q) {
        if (!done && hv[q] == bv && hi[q] == bi) {
          const int p = lane + 32 * q;
          const int h = ++head[q];
          hi[q] = h < KL ? li[p * KL + h] : -1;
          hv[q] = hi[q] >= 0 ? lv[p * KL + h] : -INFINITY;
          done = true;
        }
      }
    }
    if (lane == r) {
      my_v = bv;
      my_i = bi;
    }
  }
  return kth;
}

// ---- the tails of full narrow lists (narrow_tails) --------------------------------------------------------------
// Speculative lists (KL < K): a FULL list whose last entry is at or above the merged K-th value `kth` may have dropped
// members of (or ties with) the top-K.  Every such live list of the lane gets its bit in the warp's doubt mask `dmask`
// (null: no marks) and sets `doubt`.  Returns the lane-local largest last entry of a full live list (-inf: none) --
// what the producer of a class shard reports as its bound when the certificate is left to the owner of the row.
// K-entry lists drop nothing that could matter: -inf, no marks.
template <int kMaxListsPerLane>
__device__ __forceinline__ float narrow_tails(const float* lv, const int32_t* li, int KL, int K,
                                              const bool (&live)[kMaxListsPerLane], int lane, float kth, uint32_t* dmask,
                                              bool& doubt) {
  float tailmax = -INFINITY;
  if (KL < K) {
#pragma unroll
    for (int q = 0; q < kMaxListsPerLane; ++q) {
      const int p = lane + 32 * q;
      if (live[q] && li[p * KL + KL - 1] >= 0) {
        tailmax = fmaxf(tailmax, lv[p * KL + KL - 1]);
        if (dmask && lv[p * KL + KL - 1] >= kth) {
          doubt = true;
          atomicOr(&dmask[p >> 5], 1u << (p & 31));
        }
      }
    }
  }
  return tailmax;
}

// kMaxListsPerLane: 4 covers P <= 128 lists per row, 10 covers P <= 320 (one list per epilogue warp of
// every CTA when a single row tile is spread over all 148 SMs)
template <int kMaxListsPerLane>
__global__ void __launch_bounds__(kMergeWarps * 32, 7)  // (the cold repair functions must not set the register count)
topk_merge_kernel(const __grid_constant__ MergeArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ int s_hits[HGR_NUM_HITS];
  __shared__ uint32_t s_dmask[kMergeWarps][kDoubtWords];
  if (threadIdx.x < HGR_NUM_HITS) s_hits[threadIdx.x] = 0;
  if (threadIdx.x < kMergeWarps * kDoubtWords) (&s_dmask[0][0])[threadIdx.x] = 0;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KL = a.KL, K = a.K;
  const int64_t row0 = static_cast<int64_t>(blockIdx.x) * kMergeWarps;
  const int slots = static_cast<int>(a.P);                   // list slots per row in shared memory
  float* s_val = reinterpret_cast<float*>(smem_raw);         // [kMergeWarps][slots][KL]
  int32_t* s_idx = reinterpret_cast<int32_t*>(s_val + kMergeWarps * slots * KL);
  const int64_t pstride = a.part_stride > 0 ? a.part_stride : a.B * KL;

  // ---- stage: [list][row][KL] global -> [row][list][KL] shared
  for (int r = 0; r < kMergeWarps; ++r) {
    const int64_t row = row0 + r;
    if (row >= a.B) break;
    const int cnt = row_lists(a, row);
    const int n = cnt * KL;
    for (int e = threadIdx.x; e < n; e += kMergeWarps * 32) {
      const int p = e / KL, k = e - p * KL;
      const int64_t g = p * pstride + row * KL + k;
      s_val[(r * slots + p) * KL + k] = a.part_val[g];
      s_idx[(r * slots + p) * KL + k] = a.part_idx[g];
    }
  }
  __syncthreads();

  const int64_t row = row0 + warp;
  if (row < a.B) {
    const int cnt = row_lists(a, row);
    const float* lv = s_val + warp * slots * KL;
    const int32_t* li = s_idx + warp * slots * KL;

    bool live[kMaxListsPerLane];
#pragma unroll
    for (int q = 0; q < kMaxListsPerLane; ++q) live[q] = lane + 32 * q < cnt;
    float my_v;  // lane r keeps rank r of the result
    int32_t my_i;
    const float kth = merge_heads<kMaxListsPerLane>(lv, li, KL, K, live, lane, my_v, my_i);
    bool doubt = false;
    const float tailmax = narrow_tails<kMaxListsPerLane>(lv, li, KL, K, live, lane, kth, s_dmask[warp], doubt);
    finish_row(a, row, lane, my_v, my_i, doubt, s_dmask[warp], cnt, s_hits, tailmax);
  }
  flush_hits(a, s_hits, threadIdx.x);
}

// ---- selection merge (few candidates per row) -----------------------------------------------------------------
// When a row has at most 32 * NPL candidates in all its lists, the K rounds of the P-way merge above (two warp
// reductions, a ballot and a dependent shared-memory read per round) are replaced by a SELECTION: every lane keeps
// NPL candidates in registers as order-preserving integer keys, the K-th largest key is found by bisection (one
// compare per candidate and one REDUX.ADD per step, ~24 steps for cosines), ties at the cut are resolved by
// ascending item, and the <= K winners are compacted and ranked by counting.  ~4x fewer instructions per row; the
// result is the same (value desc, item asc) order.
template <int NPL>
__global__ void __launch_bounds__(kMergeWarps * 32, 7)  // (the cold repair functions must not set the register count)
topk_select_kernel(const __grid_constant__ MergeArgs a) {
  HGR_PLACE_ENTER();
  __shared__ int s_hits[HGR_NUM_HITS];
  __shared__ unsigned long long s_win[kMergeWarps][32];
  __shared__ uint32_t s_dmask[kMergeWarps][kDoubtWords];
  if (threadIdx.x < HGR_NUM_HITS) s_hits[threadIdx.x] = 0;
  if (threadIdx.x < kMergeWarps * kDoubtWords) (&s_dmask[0][0])[threadIdx.x] = 0;
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KL = a.KL, K = a.K;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp;
  const int64_t pstride = a.part_stride > 0 ? a.part_stride : a.B * KL;
  if (row < a.B) {
    const int cnt = row_lists(a, row);
    const int N = cnt * KL;

    uint32_t key[NPL];   // 0 = empty slot; larger key <=> larger value
    int32_t item[NPL];
    bool tail[NPL];      // last entry of a full list (certificate)
    float val[NPL];
    // all loads first, unconditionally (an out-of-range slot re-reads entry 0): 2 * NPL independent requests in
    // flight instead of a chain of dependent L2 round trips
#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      const int e = lane + 32 * s;
      const int p = e < N ? e / KL : 0, k = e < N ? e - p * KL : 0;
      const int64_t g = N > 0 ? p * pstride + row * KL + k : 0;
      item[s] = (N > 0) ? __ldg(a.part_idx + g) : -1;
      val[s] = (N > 0) ? __ldg(a.part_val + g) : 0.f;
      tail[s] = (k == KL - 1);
    }
#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      const bool ok = (lane + 32 * s < N) && item[s] >= 0;
      key[s] = ok ? order_key(val[s]) : 0u;
      item[s] = ok ? item[s] : -1;
      tail[s] = ok && tail[s];
    }
    uint32_t kmax = 0, kmin = 0xFFFFFFFFu;
    int nvalid = 0;
#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      kmax = key[s] > kmax ? key[s] : kmax;
      kmin = (key[s] != 0 && key[s] < kmin) ? key[s] : kmin;
      nvalid += key[s] != 0;
    }
    kmax = __reduce_max_sync(0xffffffffu, kmax);
    kmin = __reduce_min_sync(0xffffffffu, kmin);
    nvalid = __reduce_add_sync(0xffffffffu, nvalid);
    const int ksel = nvalid < K ? nvalid : K;

    float my_v = -INFINITY;
    int32_t my_i = -1;
    bool doubt = false;
    float tailmax = -INFINITY;
#pragma unroll
    for (int s = 0; s < NPL; ++s)
      if (tail[s]) tailmax = fmaxf(tailmax, val[s]);
    if (ksel > 0) {
      // largest T with #{key >= T} >= ksel
      uint32_t lo = kmin, hi = kmax;
      while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo + 1) >> 1);
        int c = 0;
#pragma unroll
        for (int s = 0; s < NPL; ++s) c += key[s] >= mid;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= ksel) lo = mid;
        else hi = mid - 1;
      }
      const uint32_t T = lo;
      bool sel[NPL];
      int above = 0;
#pragma unroll
      for (int s = 0; s < NPL; ++s) {
        sel[s] = key[s] > T;
        above += sel[s];
        if (tail[s] && key[s] >= T) {
          doubt = true;
          const int p = (lane + 32 * s) / KL;
          atomicOr(&s_dmask[warp][p >> 5], 1u << (p & 31));
        }
      }
      above = __reduce_add_sync(0xffffffffu, above);
      for (int need = ksel - above; need > 0; --need) {  // ties at the cut: ascending item
        uint32_t best = 0xFFFFFFFFu;
#pragma unroll
        for (int s = 0; s < NPL; ++s)
          if (key[s] == T && !sel[s] && static_cast<uint32_t>(item[s]) < best) best = static_cast<uint32_t>(item[s]);
        best = __reduce_min_sync(0xffffffffu, best);
#pragma unroll
        for (int s = 0; s < NPL; ++s)
          if (key[s] == T && !sel[s] && static_cast<uint32_t>(item[s]) == best) sel[s] = true;
      }
      // compact the winners (one per lane), rank them by counting on (key desc, item asc)
      int base = 0;
#pragma unroll
      for (int s = 0; s < NPL; ++s) {
        const unsigned b = __ballot_sync(0xffffffffu, sel[s]);
        if (sel[s]) {
          const int pos = base + __popc(b & ((1u << lane) - 1u));
          if (pos < 32)
            s_win[warp][pos] = winner_word(key[s], static_cast<uint32_t>(item[s]));
        }
        base += __popc(b);
      }
      rank_winners(s_win[warp], ksel, lane, my_v, my_i);
    }
    finish_row(a, row, lane, my_v, my_i, doubt, s_dmask[warp], cnt, s_hits, tailmax);
  }
  flush_hits(a, s_hits, threadIdx.x);
  HGR_PLACE_LEAVE(kMerge);
}

// ---- ranking merge (very few candidates per row) ------------------------------------------------------------------
// Up to 32 * NPL <= 96 candidates per row -- the class-sharded head at B = 4096: 4-6 lists of 10-16 entries for each of
// 4,096 rows, where the bisection of topk_select_kernel (~1,500 instructions per row, 66 % issue utilisation: it
// competes with the persistent GEMM of the next batch for SMs) is the expensive part.  Here every candidate is packed
// into one 64-bit word (order key << 32 | ~item: larger word = better candidate, ties by ascending item) and staged in
// shared memory list by list; the lists are SORTED, so the output position of a candidate is its position in its own
// list plus, for every other list, the number of entries that beat it -- a 5-step binary search each.
// ~350 instructions per row at 40 candidates.  Same result, same order as the other merge kernels.  Requires every
// list sorted by (value desc, item asc) -- true for the lists the scoring kernel writes.
template <int NPL>
__global__ void __launch_bounds__(kMergeWarps * 32, 7)
topk_rank_kernel(const __grid_constant__ MergeArgs a) {
  __shared__ int s_hits[HGR_NUM_HITS];
  __shared__ unsigned long long s_list[kMergeWarps][32 * NPL];
  __shared__ unsigned long long s_win[kMergeWarps][32];
  __shared__ uint32_t s_dmask[kMergeWarps][kDoubtWords];
  if (threadIdx.x < HGR_NUM_HITS) s_hits[threadIdx.x] = 0;
  if (threadIdx.x < kMergeWarps * kDoubtWords) (&s_dmask[0][0])[threadIdx.x] = 0;
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KL = a.KL, K = a.K;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp;
  const int64_t pstride = a.part_stride > 0 ? a.part_stride : a.B * KL;
  if (row < a.B) {
    const int cnt = row_lists(a, row);
    const int N = cnt * KL;

    unsigned long long w[NPL];   // 0 = empty slot
    int32_t item[NPL];
    float val[NPL];
    int lp[NPL], lk[NPL];        // list / position of my candidate
#pragma unroll
    for (int s = 0; s < NPL; ++s) {   // all loads first (an out-of-range slot re-reads entry 0)
      const int e = lane + 32 * s;
      lp[s] = e < N ? e / KL : 0;
      lk[s] = e < N ? e - lp[s] * KL : 0;
      const int64_t g = N > 0 ? lp[s] * pstride + row * KL + lk[s] : 0;
      item[s] = (N > 0) ? __ldg(a.part_idx + g) : -1;
      val[s] = (N > 0) ? __ldg(a.part_val + g) : 0.f;
    }
    int nvalid = 0;
    float tailmax = -INFINITY;
    bool tail[NPL];
#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      const bool ok = (lane + 32 * s < N) && item[s] >= 0;
      w[s] = ok ? winner_word(order_key(val[s]), static_cast<uint32_t>(item[s])) : 0ull;
      tail[s] = ok && lk[s] == KL - 1;
      if (tail[s]) tailmax = fmaxf(tailmax, val[s]);
      nvalid += ok;
      s_list[warp][lane + 32 * s] = w[s];
    }
    __syncwarp();
    nvalid = __reduce_add_sync(0xffffffffu, nvalid);
    const int ksel = nvalid < K ? nvalid : K;

#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      int rank = lk[s];
#pragma unroll 4
      for (int q = 0; q < cnt; ++q) {
        // entries of list q that come before mine: strictly larger words; an identical word (the same item reported
        // twice) counts when it sits in an earlier list
        const unsigned long long bar = w[s] - (q < lp[s] ? 1ull : 0ull);
        const unsigned long long* lq = &s_list[warp][q * KL];
        int lo = 0, hi = KL;
        while (lo < hi) {   // <= 6 steps, warp-uniform trip count would need KL a power of two: plain loop
          const int mid = (lo + hi) >> 1;
          if (lq[mid] > bar) lo = mid + 1;
          else hi = mid;
        }
        rank += q == lp[s] ? 0 : lo;
      }
      if (w[s] != 0ull && rank < 32) s_win[warp][rank] = w[s];
    }
    __syncwarp();
    float my_v = -INFINITY;
    int32_t my_i = -1;
    bool doubt = false;
    if (ksel > 0) {
      if (lane < ksel) {
        const unsigned long long x = s_win[warp][lane];
        my_v = winner_value(x);
        my_i = winner_item(x);
      }
      const uint32_t T = static_cast<uint32_t>(s_win[warp][ksel - 1] >> 32);   // key of the K-th winner
#pragma unroll
      for (int s = 0; s < NPL; ++s) {
        if (tail[s] && static_cast<uint32_t>(w[s] >> 32) >= T) {
          doubt = true;
          atomicOr(&s_dmask[warp][lp[s] >> 5], 1u << (lp[s] & 31));
        }
      }
    }
    finish_row(a, row, lane, my_v, my_i, doubt, s_dmask[warp], cnt, s_hits, tailmax);
  }
  flush_hits(a, s_hits, threadIdx.x);
}

// ---- candidate-list merge (floor-sketch epilogue) ---------------------------------------------------------------
// The lists of a row are short, UNSORTED and of different lengths (sk_cnt).  One warp per row: the lists are gathered
// into shared memory (lane = list, one 8-byte entry per step), the K-th largest order key is found by bisection over
// the gathered entries (stops early when a cut holds exactly K), ties at the cut resolve by ascending bank row, and the
// <= K winners are ranked by counting on (key desc, bank row asc) -- the same documented order as the other paths.
__global__ void __launch_bounds__(kMergeWarps * 32, 7)  // (the cold repair functions must not set the register count)
topk_merge_counts_kernel(const __grid_constant__ MergeArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ int s_hits[HGR_NUM_HITS];
  __shared__ unsigned long long s_win[kMergeWarps][32];
  if (threadIdx.x < HGR_NUM_HITS) s_hits[threadIdx.x] = 0;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = a.K, cap = a.sk_cap;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp;
  uint2* cand = reinterpret_cast<uint2*>(smem_raw) + static_cast<size_t>(warp) * a.P * cap;
  if (row < a.B) {
    const int lists = row_lists(a, row);
    int N = 0;
    for (int l0 = 0; l0 < lists; l0 += 32) {
      const int l = l0 + lane;
      int c = l < lists ? __ldg(a.sk_cnt + static_cast<int64_t>(l) * a.B + row) : 0;
      c = c < 0 ? 0 : (c > cap ? cap : c);
      int incl = c;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
      }
      const uint2* src = a.sk_part + (static_cast<int64_t>(l < lists ? l : 0) * a.B + row) * cap;
      uint2* dst = cand + N + incl - c;
      const int maxc = __reduce_max_sync(0xffffffffu, c);
      for (int k = 0; k < maxc; ++k)
        if (k < c) dst[k] = __ldg(src + k);
      N += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    // keys of this lane's entries: lane, lane + 32, ...
    uint32_t kmax = 0, kmin = 0xFFFFFFFFu;
    for (int e = lane; e < N; e += 32) {
      const uint32_t k = order_key(__uint_as_float(cand[e].x));
      cand[e].x = k;   // keep the key: the value is recovered from it
      kmax = k > kmax ? k : kmax;
      kmin = k < kmin ? k : kmin;
    }
    __syncwarp();
    kmax = __reduce_max_sync(0xffffffffu, kmax);
    kmin = __reduce_min_sync(0xffffffffu, kmin);
    const int ksel = N < K ? N : K;
    float my_v = -INFINITY;
    int32_t my_i = -1;
    if (ksel > 0) {
      // largest T with #{key >= T} >= ksel; done as soon as a cut holds exactly ksel entries
      uint32_t lo = kmin, hi = kmax;
      int c_lo = N;
      while (lo < hi && c_lo != ksel) {
        const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
        int c = 0;
        for (int e = lane; e < N; e += 32) c += cand[e].x >= mid;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= ksel) {
          lo = mid;
          c_lo = c;
        } else {
          hi = mid - 1u;
        }
      }
      const uint32_t T = lo;
      int need = 0;   // tied entries at T still to be taken (ascending bank row)
      if (c_lo != ksel) {
        int above = 0;
        for (int e = lane; e < N; e += 32) above += cand[e].x > T;
        need = ksel - __reduce_add_sync(0xffffffffu, above);
      }
      uint32_t tie_floor = 0;   // tied bank rows below this one are already taken
      bool tie_any = false;
      int base = 0;
      // winners above the cut (or at it, when the cut is exact), compacted one per lane
      for (int e0 = 0; e0 < N; e0 += 32) {
        const int e = e0 + lane;
        const bool sel = e < N && (c_lo == ksel ? cand[e].x >= T : cand[e].x > T);
        const unsigned b = __ballot_sync(0xffffffffu, sel);
        if (sel) {
          const int pos = base + __popc(b & ((1u << lane) - 1u));
          if (pos < 32) s_win[warp][pos] = winner_word(cand[e].x, cand[e].y);
        }
        base += __popc(b);
      }
      for (; need > 0; --need) {
        uint32_t best = 0xFFFFFFFFu;
        for (int e = lane; e < N; e += 32)
          if (cand[e].x == T && (!tie_any || cand[e].y > tie_floor) && cand[e].y < best) best = cand[e].y;
        best = __reduce_min_sync(0xffffffffu, best);
        if (lane == 0 && base < 32) s_win[warp][base] = winner_word(T, best);
        ++base;
        tie_floor = best;
        tie_any = true;
      }
      rank_winners(s_win[warp], ksel, lane, my_v, my_i);
    }
    finish_row(a, row, lane, my_v, my_i, false, nullptr, 0, s_hits);
  }
  flush_hits(a, s_hits, threadIdx.x);
}

// ---- per-split merge (hgr_score_topk_splits) --------------------------------------------------------------------
// The lists of a row on the grouped schedule never cross a group, so the lists of the row's groups in split s cover
// exactly the columns of s.  One warp per row stages all the row's lists in shared memory, then for every split runs
// merge_heads over that split's lists only, certifies the result against the split's own K-th value (narrow_tails)
// and, for an uncertified (row, split), re-scans that split's doubtful lists exactly (repair_lists).
constexpr int kSplitDoubtWords = 4;   // bit per list, up to 128 lists per row

// Per-split Hit@k and row counters of a CTA: cnt[c] (= s_cnt[s][c]) counts Hit@hit_cut(c), cnt[HGR_NUM_HITS] the rows
// whose label is a class of split s.  count_split_row: one such row, lane r holding rank r (node id `gid`, -1: none)
// of its list of s.
__device__ __forceinline__ void count_split_row(unsigned int* cnt, int lane, int K, int32_t gid, int32_t target) {
  const unsigned m = __ballot_sync(0xffffffffu, lane < K && gid >= 0 && gid == target);
  if (lane == 0) {
    atomicAdd(&cnt[HGR_NUM_HITS], 1u);
    if (m != 0) {
      const int pos = __ffs(m) - 1;
#pragma unroll
      for (int c = 0; c < HGR_NUM_HITS; ++c)
        if (pos < hit_cut(c)) atomicAdd(&cnt[c], 1u);
    }
  }
}
// The CTA's counters of the S splits into counts[S][HGR_NUM_HITS + 1] (null: none).  `tid` = threadIdx.x (flush_hits).
__device__ __forceinline__ void flush_split_counts(const unsigned int (*s_cnt)[HGR_NUM_HITS + 1], int S, int64_t* counts,
                                                   int tid) {
  __syncthreads();
  if (counts) {
    for (int i = tid; i < S * (HGR_NUM_HITS + 1); i += blockDim.x) {
      const unsigned int v = (&s_cnt[0][0])[i];
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(counts) + i, static_cast<unsigned long long>(v));
    }
  }
}

// kScatter (hgr_score_topk_splits_scatter_bounded, producer of the class-sharded head): no local certificate or repair;
// split s of the row goes to its owner's slot next to the bound of what the split's full narrow lists dropped.
template <int kMaxListsPerLane, bool kScatter>
__global__ void __launch_bounds__(kMergeWarps * 32, 4)  // (the cold repair function must not set the register count)
topk_split_merge_kernel(const __grid_constant__ SplitMergeArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ unsigned int s_cnt[kMaxSplits][HGR_NUM_HITS + 1];
  __shared__ uint32_t s_dmask[kMergeWarps][kSplitDoubtWords];
  for (int i = threadIdx.x; i < kMaxSplits * (HGR_NUM_HITS + 1); i += blockDim.x) (&s_cnt[0][0])[i] = 0u;
  if (threadIdx.x < kMergeWarps * kSplitDoubtWords) (&s_dmask[0][0])[threadIdx.x] = 0u;
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KL = a.KL, K = a.K;
  const int slots = a.sched.P;
  float* lv = reinterpret_cast<float*>(smem_raw) + warp * slots * KL;                   // [slots][KL] of this row
  int32_t* li = reinterpret_cast<int32_t*>(reinterpret_cast<float*>(smem_raw) + kMergeWarps * slots * KL) + warp * slots * KL;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp;
  if (row < a.B) {
    const int32_t mt = static_cast<int32_t>(row / a.sched.rows);
    const int cnt = group_parts(a.sched, a.groups, mt);
    for (int e = lane; e < cnt * KL; e += 32) {
      const int p = e / KL, k = e - p * KL;
      const int64_t g = (p * a.B + row) * KL + k;
      lv[e] = a.part_val[g];
      li[e] = a.part_idx[g];
    }
    // split bits of my lists: lane h holds the first slot of group h
    const int ng = a.groups.n;
    const int fs = lane < ng ? group_first_slot(a.sched, a.groups, mt, lane) : 0x7FFFFFFF;
    int grp[kMaxListsPerLane];
#pragma unroll
    for (int q = 0; q < kMaxListsPerLane; ++q) grp[q] = 0;
    for (int h = 1; h < ng; ++h) {
      const int f = __shfl_sync(0xffffffffu, fs, h);
#pragma unroll
      for (int q = 0; q < kMaxListsPerLane; ++q)
        if (lane + 32 * q >= f) grp[q] = h;
    }
    uint32_t lmask[kMaxListsPerLane];
#pragma unroll
    for (int q = 0; q < kMaxListsPerLane; ++q) lmask[q] = lane + 32 * q < cnt ? a.group_splits[grp[q]] : 0u;
    __syncwarp();
    const int32_t target = a.targets ? a.targets[row] : -1;
    const uint32_t tbits = (target >= 0 && target < a.n_nodes) ? a.node_splits[target] : 0u;

    for (int s = 0; s < a.S; ++s) {
      bool live[kMaxListsPerLane];
#pragma unroll
      for (int q = 0; q < kMaxListsPerLane; ++q) live[q] = (lmask[q] >> s) & 1u;
      float my_v;
      int32_t my_i;
      const float kth = merge_heads<kMaxListsPerLane>(lv, li, KL, K, live, lane, my_v, my_i);
      // certificate against the split's own K-th value: a full narrow list of s that ends at or above it may hide
      // members of the split's top-K (kScatter: the bound of what they dropped, no certificate)
      bool doubt = false;
      const float tailmax =
          narrow_tails<kMaxListsPerLane>(lv, li, KL, K, live, lane, kth, kScatter ? nullptr : s_dmask[warp], doubt);
      if constexpr (kScatter) {
        const float b = warp_max_f32(tailmax);
        const int64_t g = row / a.scatter.block_rows;
        const int64_t orow = row - g * a.scatter.block_rows;
        const int64_t so = s * a.split_stride;
        if (lane < K) {
          a.scatter.val[g][so + orow * K + lane] = my_i >= 0 ? my_v * a.scale : -INFINITY;
          a.scatter.idx[g][so + orow * K + lane] = my_i >= 0 ? (a.col_id ? a.col_id[my_i] : a.id_base + my_i) : -1;
        }
        if (lane == 0) a.scatter.bound[g][so + orow] = b * a.scale;
        continue;
      }
      if (__any_sync(0xffffffffu, doubt)) {
        __syncwarp();
        const Cand c = repair_cold(&a, row, lane, cnt, s, s_dmask[warp]);
        my_v = c.v;
        my_i = c.i;
        __syncwarp();
        if (lane < kSplitDoubtWords) s_dmask[warp][lane] = 0u;
        __syncwarp();
      }
      int32_t gid = -1;
      if (lane < K && my_i >= 0) gid = a.col_id ? a.col_id[my_i] : a.id_base + my_i;
      if (lane < K) {
        const int64_t o = (s * a.B + row) * K + lane;
        a.topk_val[o] = my_i >= 0 ? my_v * a.scale : -INFINITY;
        a.topk_idx[o] = gid;
      }
      if (a.counts && ((tbits >> s) & 1u)) count_split_row(s_cnt[s], lane, K, gid, target);
    }
  }
  flush_split_counts(s_cnt, a.S, a.counts, threadIdx.x);
}

// ---- per-split certified merge of the class-sharded head (hgr_topk_merge_splits_certified) -------------------------
// Owner side of hgr_score_topk_splits_scatter_bounded.  For every owned row and split s the P shard lists of s are merged
// in the order (value desc, shard asc, position in the list asc): each list is the shard's top-K of s in (value desc,
// local bank row asc) order, so the result is the top-K of s's rows concatenated in rank-major order -- what score_topk
// returns on that bank.  The merged K-th value must strictly beat every shard's bound of s; a doubtful (row, split,
// shard) is re-scanned exactly from the shard table (repair_shards).
// One warp per row; lane p holds the head of shard p's list.  Per output rank: the largest head value, the lowest lane
// among equals, and that lane advances.
__global__ void __launch_bounds__(kMergeWarps * 32)   // (a cap on the registers makes the merge spill around the call)
topk_split_cert_kernel(const __grid_constant__ SplitCertArgs a) {
  __shared__ unsigned int s_cnt[kMaxSplits][HGR_NUM_HITS + 1];
  for (int i = threadIdx.x; i < kMaxSplits * (HGR_NUM_HITS + 1); i += blockDim.x) (&s_cnt[0][0])[i] = 0u;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = a.K;
  const int P = static_cast<int>(a.P);
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kMergeWarps + warp;
  if (row < a.B) {
    const int32_t target = a.targets ? a.targets[row] : -1;
    const uint32_t tbits = (target >= 0 && target < a.n_nodes) ? a.node_splits[target] : 0u;
    for (int s = 0; s < a.S; ++s) {
      const int64_t lbase = s * a.split_stride + lane * a.part_stride + row * K;
      int head = 0;
      float hv = -INFINITY;
      int32_t hi = -1;
      if (lane < P) {
        hi = a.part_idx[lbase];
        hv = a.part_val[lbase];
      }
      float my_v = -INFINITY;
      int32_t my_i = -1;
      for (int r = 0; r < K; ++r) {
        const bool live = hi >= 0;
        const uint32_t mkey = __reduce_max_sync(0xffffffffu, live ? order_key(hv) : 0u);
        const unsigned cand = __ballot_sync(0xffffffffu, live && order_key(hv) == mkey);
        if (cand == 0u) break;                      // every list exhausted: the rest stays (-inf, -1)
        const int win = __ffs(cand) - 1;
        const float bv = __shfl_sync(0xffffffffu, hv, win);
        const int32_t bi = __shfl_sync(0xffffffffu, hi, win);
        if (lane == r) {
          my_v = bv;
          my_i = bi;
        }
        if (lane == win) {
          ++head;
          hi = head < K ? a.part_idx[lbase + head] : -1;
          hv = hi >= 0 ? a.part_val[lbase + head] : -INFINITY;
        }
      }
      // certificate: the merged K-th value strictly above every shard's bound of s (fewer than K merged: -inf, so any
      // shard that dropped something is doubtful)
      const float kth = __shfl_sync(0xffffffffu, my_i >= 0 ? my_v : -INFINITY, K - 1);
      const float bnd = lane < P ? a.part_bound[s * a.split_stride + lane * a.bound_stride + row] : -INFINITY;
      const unsigned dm = __ballot_sync(0xffffffffu, bnd > -INFINITY && bnd >= kth);
      if (dm != 0u) {
        const Cand c = repair_cold(&a, row, lane, s, dm);
        my_v = c.v;
        my_i = c.i;
      }
      if (lane < K) {
        const int64_t o = (s * a.B + row) * K + lane;
        a.topk_val[o] = my_i >= 0 ? my_v : -INFINITY;
        a.topk_idx[o] = my_i;
      }
      if (a.counts && ((tbits >> s) & 1u)) count_split_row(s_cnt[s], lane, K, my_i, target);
    }
  }
  flush_split_counts(s_cnt, a.S, a.counts, threadIdx.x);
}

// ---- cross-GPU sequencing of the peer-memory exchange ---------------------------------------------------------
// Every rank keeps `n` flag words (one per producer rank) in its exchange buffer.  After the kernel that wrote its
// candidates into the peers' buffers, a rank launches peer_signal: thread g stores the rank's running sequence
// number into ITS flag word on rank g (system-scope release; the scatter kernel finished before, stream order).
// Before merging, a rank launches peer_wait: thread g spins (system-scope acquire) until producer g's flag has
// reached the consumer's own running sequence number.  Both counters live in device memory and advance by one per
// launch, so the pair can be captured in a CUDA graph and replayed.
struct PeerFlags {
  uint32_t* p[kMaxScatterBlocks];
};

__global__ void peer_signal_kernel(const PeerFlags flags, int n, uint32_t* seq) {
  __shared__ uint32_t s_v;
  if (threadIdx.x == 0) s_v = ++(*seq);
  __syncthreads();
  if (static_cast<int>(threadIdx.x) < n) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flags.p[threadIdx.x]), "r"(s_v) : "memory");
  }
}

__global__ void peer_wait_kernel(const uint32_t* flags, int n, uint32_t* seq, unsigned long long timeout_ns) {
  __shared__ uint32_t s_v;
  if (threadIdx.x == 0) s_v = ++(*seq);
  __syncthreads();
  if (static_cast<int>(threadIdx.x) < n) {
    const uint32_t want = s_v;
    unsigned long long t0 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t got;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(got) : "l"(flags + threadIdx.x) : "memory");
      if (static_cast<int32_t>(got - want) >= 0) break;
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) {  // a peer died or the schedules diverged -- fail loudly, never hang the GPU
        printf("hgr peer_wait: producer %d stuck at %u, waiting for %u\n", static_cast<int>(threadIdx.x), got, want);
        __trap();
      }
      __nanosleep(200);
    }
  }
}

}  // namespace

int launch_peer_signal(uint32_t* const* flags, int n, uint32_t* seq, cudaStream_t stream) {
  if (n < 1 || n > kMaxScatterBlocks) return set_error(HGR_ERR_BAD_ARG, "peer signal: %d ranks outside [1, %d]", n, kMaxScatterBlocks);
  PeerFlags f{};
  for (int g = 0; g < n; ++g) f.p[g] = flags[g];
  peer_signal_kernel<<<1, 32, 0, stream>>>(f, n, seq);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_peer_wait(const uint32_t* flags, int n, uint32_t* seq, cudaStream_t stream) {
  if (n < 1 || n > kMaxScatterBlocks) return set_error(HGR_ERR_BAD_ARG, "peer wait: %d ranks outside [1, %d]", n, kMaxScatterBlocks);
  // how long a consumer waits for the slowest producer before it traps: 10 s unless HGR_PEER_TIMEOUT_MS says otherwise
  // (a rank whose host stalls longer than this between two graph launches would take the job down)
  static const unsigned long long timeout_ns = [] {
    const char* e = getenv("HGR_PEER_TIMEOUT_MS");
    const long long ms = e ? atoll(e) : 10000;
    return static_cast<unsigned long long>(ms > 0 ? ms : 10000) * 1000000ull;
  }();
  peer_wait_kernel<<<1, 32, 0, stream>>>(flags, n, seq, timeout_ns);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

// The merge that holds a row's `cand` candidates (an upper bound) in registers, or nullptr when they do not fit and
// the lists are merged from shared memory.
using RegMerge = void (*)(MergeArgs);
static RegMerge register_merge(int64_t cand, bool use_sched) {
  // (only for the scoring kernel's own lists: bank rows, sorted (value desc, row asc) by construction -- lists handed
  //  to hgr_topk_merge carry node ids, whose order among equal values is the caller's)
#ifndef HGR_NO_RANK_KERNEL   // (kernel experiments: tools/build_variant.sh norank -DHGR_NO_RANK_KERNEL topk_merge.cu)
  if (cand <= 96 && use_sched) return cand <= 64 ? topk_rank_kernel<2> : topk_rank_kernel<3>;
#endif
  if (cand <= 320) return cand <= 128 ? topk_select_kernel<4> : (cand <= 192 ? topk_select_kernel<6> : topk_select_kernel<10>);
  return nullptr;
}

#ifdef HGR_PLACEMENT
int placement_attach_merge(const place::Log& l) { return place::attach(l); }
#endif

int merge_kernel_footprint(int64_t P, int KL, int32_t* out) {
  const RegMerge kern = register_merge(P * KL, true);
  if (kern == nullptr) return set_error(HGR_ERR_UNSUPPORTED, "merge footprint: %lld x %d candidates per row", (long long)P, KL);
  cudaFuncAttributes fa;
  HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, kern));
  out[0] = kMergeWarps * 32;
  out[1] = fa.numRegs;
  out[2] = static_cast<int32_t>(fa.sharedSizeBytes);
  out[3] = 0;
  return HGR_OK;
}

int launch_topk_merge(const MergeArgs& args, cudaStream_t stream) {
  if (args.B == 0 || args.K == 0) return HGR_OK;
  if (args.sk_part != nullptr) {
    if (args.K > 32 || args.sk_cap < 1 || args.sk_cnt == nullptr)
      return set_error(HGR_ERR_BAD_ARG, "topk merge (candidate lists): K = %d / cap = %d", args.K, args.sk_cap);
    const int blocks = static_cast<int>((args.B + kMergeWarps - 1) / kMergeWarps);
    const size_t smem = static_cast<size_t>(kMergeWarps) * args.P * args.sk_cap * 8;
    if (smem > 200 * 1024) return set_error(HGR_ERR_UNSUPPORTED, "topk merge: %zu bytes of candidates per CTA", smem);
    HGR_CHECK_CUDA(cudaFuncSetAttribute(topk_merge_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    topk_merge_counts_kernel<<<blocks, kMergeWarps * 32, smem, stream>>>(args);
    HGR_CHECK_LAUNCH();
    return HGR_OK;
  }
  if (args.P > 320)
    return set_error(HGR_ERR_UNSUPPORTED, "topk merge: %lld lists per row exceed 320", (long long)args.P);
  if (args.K > HGR_TOPK_MAX || args.KL < 1)
    return set_error(HGR_ERR_UNSUPPORTED, "topk merge: K = %d / KL = %d unsupported", args.K, args.KL);
  if (args.KL < args.K && (args.X == nullptr || args.bank == nullptr || !args.use_sched))
    return set_error(HGR_ERR_BAD_ARG, "topk merge: speculative lists need X / bank / the schedule for the exact repair");
  const int blocks = static_cast<int>((args.B + kMergeWarps - 1) / kMergeWarps);
  if (const RegMerge kern = register_merge(args.P * args.KL, args.use_sched)) {
    kern<<<blocks, kMergeWarps * 32, 0, stream>>>(args);
    HGR_CHECK_LAUNCH();
    return HGR_OK;
  }
  const size_t smem = static_cast<size_t>(kMergeWarps) * args.P * args.KL * 8;
  if (smem > 200 * 1024) return set_error(HGR_ERR_UNSUPPORTED, "topk merge: %zu bytes of lists per CTA", smem);
  if (args.P <= 128) {
    if (smem > 48 * 1024)
      HGR_CHECK_CUDA(cudaFuncSetAttribute(topk_merge_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          static_cast<int>(smem)));
    topk_merge_kernel<4><<<blocks, kMergeWarps * 32, smem, stream>>>(args);
  } else {
    if (smem > 48 * 1024)
      HGR_CHECK_CUDA(cudaFuncSetAttribute(topk_merge_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          static_cast<int>(smem)));
    topk_merge_kernel<10><<<blocks, kMergeWarps * 32, smem, stream>>>(args);
  }
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

template <int kMaxListsPerLane, bool kScatter>
static int launch_split_merge_kernel(const SplitMergeArgs& args, int blocks, size_t smem, cudaStream_t stream) {
  if (smem > 48 * 1024)
    HGR_CHECK_CUDA(cudaFuncSetAttribute(topk_split_merge_kernel<kMaxListsPerLane, kScatter>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  topk_split_merge_kernel<kMaxListsPerLane, kScatter><<<blocks, kMergeWarps * 32, smem, stream>>>(args);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

int launch_topk_split_merge(const SplitMergeArgs& args, cudaStream_t stream) {
  if (args.B == 0) return HGR_OK;
  if (args.sched.P > 32 * kSplitDoubtWords)
    return set_error(HGR_ERR_UNSUPPORTED, "topk split merge: %d lists per row exceed %d", args.sched.P, 32 * kSplitDoubtWords);
  const int blocks = static_cast<int>((args.B + kMergeWarps - 1) / kMergeWarps);
  const size_t smem = static_cast<size_t>(kMergeWarps) * args.sched.P * args.KL * 8;
  if (smem > 200 * 1024) return set_error(HGR_ERR_UNSUPPORTED, "topk split merge: %zu bytes of lists per CTA", smem);
  const bool scatter = args.scatter.n_blocks > 0;
  if (args.sched.P <= 64)
    return scatter ? launch_split_merge_kernel<2, true>(args, blocks, smem, stream)
                   : launch_split_merge_kernel<2, false>(args, blocks, smem, stream);
  return scatter ? launch_split_merge_kernel<4, true>(args, blocks, smem, stream)
                 : launch_split_merge_kernel<4, false>(args, blocks, smem, stream);
}

int launch_topk_split_merge_certified(const SplitCertArgs& args, cudaStream_t stream) {
  if (args.B == 0) return HGR_OK;
  const int blocks = static_cast<int>((args.B + kMergeWarps - 1) / kMergeWarps);
  topk_split_cert_kernel<<<blocks, kMergeWarps * 32, 0, stream>>>(args);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace hgr
