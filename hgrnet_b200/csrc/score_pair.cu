// Kernel (2): image x class cosine logits on tcgen05 with the per-row running top-K fused into the epilogue -- the
// B x C logit matrix never reaches HBM.  Two CTAs of a cluster (one TPC) share every MMA: tcgen05.mma.cta_group::2
// with M = 256.  The same main loop with a store epilogue backs hgr_logits_dense.
//
// Reference: `feats @ self.zsl_weights.T` (model/clip_tree.py:331), `logits[:, test_index]` +
// `.topk(20, 1, True, True)` (main.py:136-138); id mapping / hit test (main.py:139-147) run in topk_merge.cu.
//
// Why: a single-CTA 128 x 256 tile needs (128 + 256) x 64 x 2 B = 48 KB of operands per K block,
// 96 B/clk/SM at the tensor core's issue rate, and the L2 -> SM path of this chip delivers ~50
// B/clk/SM (measured: the single-CTA kernel with a null epilogue tops out at 14.4 TB/s of TMA
// reads, profiles/).  In a pair each CTA contributes its own 128 image rows (A) but only HALF of
// the bank sub-tile (B): 32 KB per K block per CTA for the same 128 x 256 outputs per CTA.
//
// Layout per CTA: A stage [128 x 64] bf16 (own rows), B stage [<=128 x 64] (leader: bank rows
// [col0, col0 + n/2), peer: [col0 + n/2, col0 + n)), both 128B-swizzled; TMEM 2 x 256 columns,
// each CTA holding the accumulators of its own 128 rows x all n columns.
// Protocol: both producers signal the LEADER's `full` barrier (cp.async.bulk.tensor
// .cta_group::2); the leader's single MMA thread commits with a cluster multicast to the `empty`
// and `tmem_full` barriers of both CTAs; the epilogue warps of both CTAs arrive on the leader's
// `tmem_empty`.  Epilogues: umma_common.cuh (deferred-insert lists), sketch_epi.cuh (floor sketch); work split: sched.cuh.
#include "placement.cuh"
#include "sketch_epi.cuh"
#include "umma_common.cuh"

namespace hgr {
namespace umma {
namespace {

constexpr int kPairStagesMax = 6;
constexpr int kPairBBytes = (kSubN / 2) * kBlockK * 2;     // 16 KB: half of the bank sub-tile
constexpr int kPairStageBytes = kABytes + kPairBBytes;     // 32 KB
constexpr int kDenseTileFloats = 32 * 33;                  // dense epilogue: one padded 32x32 transpose tile per warp

struct PairCtl {
  uint64_t full[kPairStagesMax];   // leader's copy is the one in use
  uint64_t empty[kPairStagesMax];  // per CTA, signalled by the leader's multicast commit
  uint64_t tmem_full[2];           // per CTA, multicast commit
  uint64_t tmem_empty[2];          // leader's copy: arrivals from the epilogue warps of both CTAs
  uint32_t tmem_base;
};

// What an epilogue needs of a CTA, read by the kernel (launch bounds, shared-memory carve-up, barrier counts) and by
// its launcher (threads, dynamic shared memory, opt-in limit).
template <int EPI, int KL = 8>
struct EpiRes {
  static constexpr bool kTopk = EPI == kEpiTopkDefer || EPI == kEpiTopkGroups;
  static constexpr int kQueueLen = defer_queue_len<KL>();     // top-K epilogues: candidate queue entries per thread
  static constexpr bool kQueue = kTopk || EPI == kEpiSketch;   // a candidate queue per thread
  // one warp per TMEM lane quarter; the dense epilogue has two, which take alternate chunks of every sub-tile
  static constexpr int kWarps = EPI == kEpiDense ? 8 : 4;
  static constexpr int kThreads = 64 + 32 * kWarps;           // + the TMA and the MMA warp
  static constexpr int kStagingBytes = EPI == kEpiSketch ? kSkQueueBytes
                                     : kTopk ? (kQueueLen + 1) * kDeferStride
                                     : EPI == kEpiDense ? kWarps * kDenseTileFloats * 4 : 0;
  // Operand stages: as many 32 KB stages as fit beside the staging memory (measured: 4 stages cost ~2 us of main loop
  // at cfg 2, and leaving room for co-resident small kernels that way bought nothing).  With narrow lists the shorter
  // queue (defer_queue_len) leaves room for a normalise and two merge CTAs beside a 5-stage CTA instead.
  static constexpr int kMaxStages = kQueue ? 5 : 6;
  static constexpr int kTmemEmptyArrivals = 2 * kWarps;       // every epilogue warp of both CTAs
  static constexpr size_t smem_bytes(int stages) {
    return 1024 + static_cast<size_t>(stages) * kPairStageBytes + kStagingBytes + sizeof(PairCtl);
  }
  // Run-time stage count (Params::stages).  Large batches use ONE stage less than fits: their main loop does not
  // notice (measured at B = 4096: 82.9 / 56.1 / 40.1 us either way), and the 32 KB left free let a neighbouring
  // stream's small kernels (normalise, merge, flags) share the SM with a resident GEMM CTA instead of waiting for it
  // (class-sharded pipeline: -5 % per step).  At cfg 2 (B = 512) the fifth stage is worth 0.7 us, so it stays.
  static int stages(int64_t B) { return kQueue && B >= 2048 ? kMaxStages - 1 : kMaxStages; }
};
static_assert(EpiRes<kEpiSketch>::kWarps * 32 * 8 == kSkStride &&
              EpiRes<kEpiTopkDefer>::kWarps * 32 * 8 == kDeferStride, "queue stride = one entry per epilogue thread");

// The walk of a worker over its chunk: the plain schedule, or the grouped one (kEpiTopkGroups).
template <bool kGroups>
struct WalkerOf {
  using type = TileWalker;
  __device__ __forceinline__ static TileWalker make(const Params& p, int pair) { return TileWalker(p.sched, pair, p.C); }
};
template <>
struct WalkerOf<true> {
  using type = GroupWalker;
  __device__ __forceinline__ static GroupWalker make(const Params& p, int pair) {
    return GroupWalker(p.sched, pair, p.groups);
  }
};

// TMA producer (warp 0 of both CTAs; convergent warp, elected issue -- see ptx.cuh): per K block this CTA's 128 image
// rows and its half of the bank sub-tile, both signalled on the LEADER's `full` barrier.
template <bool kGroups>
__device__ __forceinline__ void produce(const CUtensorMap* map_x, const CUtensorMap* map_bank, const Params& p,
                                        PairCtl* ctl, uint8_t* stage_base, uint32_t rank, int pair) {
  const uint64_t pol = ptx::policy_evict_last();
  auto walk = WalkerOf<kGroups>::make(p, pair);
  SubTile t;
  int stage = 0;
  uint32_t phase = 0;
  while (walk.next(t)) {
    const int half = t.n >> 1;                                   // bank rows this CTA feeds
    const int nbox = (half + kBBoxRows - 1) / kBBoxRows;
    const int row0 = t.mt * (2 * kTileM) + static_cast<int>(rank) * kTileM;
    const int bcol0 = t.col0 + static_cast<int>(rank) * half;
    for (int kb = 0; kb < p.num_k_blocks; ++kb) {
      ptx::mbar_wait(&ctl->empty[stage], phase ^ 1u);
      uint8_t* sa = stage_base + stage * kPairStageBytes;
      uint8_t* sb = sa + kABytes;
      const uint32_t full_leader = ptx::mapa_shared(ptx::smem_u32(&ctl->full[stage]), 0);
      if (ptx::elect_one()) {
        if (rank == 0) ptx::mbar_arrive_expect_tx(&ctl->full[stage], 2 * (kABytes + nbox * kBBoxBytes));
        ptx::tma_load_2d_cg2(sa, map_x, full_leader, kb * kBlockK, row0, pol);
        for (int b = 0; b < nbox; ++b)
          ptx::tma_load_2d_cg2(sb + b * kBBoxBytes, map_bank, full_leader, kb * kBlockK, bcol0 + b * kBBoxRows, pol);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  }
}

// MMA issuer (warp 1 of the leader CTA; convergent warp, elected issue): M = 256 over both CTAs, accumulators
// alternate between the two TMEM buffers.
template <bool kGroups>
__device__ __forceinline__ void issue_mma(const Params& p, PairCtl* ctl, uint8_t* stage_base, uint32_t tmem_base,
                                          int pair, int lane) {
  auto walk = WalkerOf<kGroups>::make(p, pair);
  SubTile t;
  int stage = 0;
  uint32_t phase = 0;
  int it = 0;
  const uint32_t empty0 = ptx::smem_u32(&ctl->empty[0]);
  while (walk.next(t)) {
    const int buf = it & 1;
    ptx::mbar_wait(&ctl->tmem_empty[buf], ((it >> 1) & 1) ^ 1u);
    ptx::tc_fence_after();
    if (it < 3 && lane == 0) stamp(p, 21 + it);  // accumulator buffer granted for sub-tile `it`
    const uint32_t d_tmem = tmem_base + buf * kSubN;
    const uint32_t idesc = ptx::umma_idesc_bf16(2 * kTileM, t.n);
    for (int kb = 0; kb < p.num_k_blocks; ++kb) {
      ptx::mbar_wait(&ctl->full[stage], phase);
      ptx::tc_fence_after();
      if (it == 0 && kb == 0 && lane == 0) stamp(p, 2);  // first operands landed
      const uint32_t a_addr = ptx::smem_u32(stage_base + stage * kPairStageBytes);
      const uint32_t a_lo = ptx::desc_lo_sw128(a_addr), b_lo = ptx::desc_lo_sw128(a_addr + kABytes);
      if (ptx::elect_one()) {
#pragma unroll
        for (int k = 0; k < kBlockK / kUmmaK; ++k)
          ptx::umma_bf16_cg2_lo(d_tmem, a_lo + k * (kUmmaK * 2 / 16), b_lo + k * (kUmmaK * 2 / 16), idesc,
                                (kb | k) != 0 ? 1u : 0u);
        ptx::umma_commit_cg2_mc_addr(empty0 + stage * 8, 0x3);  // frees this stage in both CTAs
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
    if (ptx::elect_one()) ptx::umma_commit_cg2_mc(&ctl->tmem_full[buf], 0x3);  // accumulators of both CTAs complete
    __syncwarp();
    ++it;
  }
  if (lane == 0) stamp(p, 3);  // last MMA issued
}

// An epilogue warp: thread = TMEM lane = image row of its CTA's 128, one lane quarter per warp (warp & 3).
struct EpiWarp {
  PairCtl* ctl;
  uint32_t tmem_base;
  uint32_t rank;   // 0 = leader
  int pair;        // worker of the schedule
  int warp, lane;
  __device__ __forceinline__ int epi_tid() const { return (warp - kEpiWarp0) * 32 + lane; }
  __device__ __forceinline__ int row_in_tile() const { return static_cast<int>(rank) * kTileM + (warp & 3) * 32 + lane; }
  // this warp's lane quarter of accumulator buffer `buf`
  __device__ __forceinline__ uint32_t taddr(int buf) const {
    return tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + buf * kSubN;
  }
  // accumulators of sub-tile `it` complete (every warp observes every phase: a skipped one would alias on the parity)
  __device__ __forceinline__ void wait_full(int it) const {
    ptx::mbar_wait(&ctl->tmem_full[it & 1], (it >> 1) & 1);
    ptx::tc_fence_after();
  }
  // this warp's share of accumulator buffer `buf` is drained: tell the leader's MMA thread
  __device__ __forceinline__ void release(int buf) const {
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (rank == 0) ptx::mbar_arrive(&ctl->tmem_empty[buf]);
      else ptx::mbar_arrive_cluster(ptx::mapa_shared(ptx::smem_u32(&ctl->tmem_empty[buf]), 0));
    }
  }
};

// First element of the partial list [slot][row][KL] of this worker's segment of row tile mt.
__device__ __forceinline__ int64_t list_offset(const Params& p, int pair, int mt, int64_t row) {
  return (static_cast<int64_t>(pair - p.sched.first_cta(mt)) * p.B + row) * p.KL;
}

// End of an epilogue warp: timeline stamp and the cycle accounting of the CTA's first epilogue warp (tools/timeline.py).
__device__ __forceinline__ void epi_done(const Params& p, const EpiClock& ck, int epi_tid) {
  if (epi_tid == 0) stamp(p, 12);  // epilogue done
  if (ck.on && blockIdx.x < 256) {
    unsigned long long* tl = p.timeline + blockIdx.x * kTimelineSlots;
    tl[16] = ck.wait, tl[17] = ck.warm, tl[18] = ck.ld, tl[19] = ck.scan, tl[20] = ck.drain;
  }
}

// ===================== epilogue: dense logits (hgr_logits_dense) =====================
// Two warps per lane quarter take alternate chunks; each transposes its 32 rows x 32 columns through a padded
// shared-memory tile, so that every store instruction writes 128 contiguous bytes of ONE row.
__device__ __forceinline__ void epi_dense(const Params& p, const EpiWarp& w, float* staging) {
  const int member = (w.warp - kEpiWarp0) >> 2;   // which of the quarter's two warps
  float* tile = staging + (w.warp - kEpiWarp0) * kDenseTileFloats;
  TileWalker walk(p.sched, w.pair, p.C);
  SubTile t;
  int it = 0;
  while (walk.next(t)) {
    const int buf = it & 1;
    const int64_t row = static_cast<int64_t>(t.mt) * (2 * kTileM) + w.row_in_tile();
    w.wait_full(it);
    const uint32_t taddr = w.taddr(buf);
    for (int c0 = member * kChunk; c0 < t.nvalid; c0 += 2 * kChunk) {
      uint32_t r[kChunk];
      ptx::tmem_ld_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      const int nv = t.nvalid - c0;
#pragma unroll
      for (int j = 0; j < kChunk; ++j) tile[w.lane * 33 + j] = __uint_as_float(r[j]) * p.scale;
      __syncwarp();
      const int64_t row_base = row - w.lane;
      float* o = p.dense_out + row_base * p.ldo + t.col0 + c0 + w.lane;
      const int nrows = p.B - row_base < 32 ? static_cast<int>(p.B - row_base) : 32;
      if (w.lane < nv) {
#pragma unroll 8
        for (int rr = 0; rr < nrows; ++rr) o[static_cast<int64_t>(rr) * p.ldo] = tile[rr * 33 + w.lane];
      }
      __syncwarp();
    }
    w.release(buf);
    ++it;
  }
}

// ===================== epilogue: null (kVarNull: the main loop's ceiling; NOT a top-k) =====================
// One running maximum per row, written as a one-entry list per segment: the least work that still reads every value.
__device__ __forceinline__ void epi_null(const Params& p, const EpiWarp& w) {
  const int epi_tid = w.epi_tid();
  TileWalker walk(p.sched, w.pair, p.C);
  SubTile t;
  float acc = -INFINITY;
  int it = 0;
  EpiClock ck(p.timeline != nullptr && epi_tid == 0);
  while (walk.next(t)) {
    const int buf = it & 1;
    const int64_t row = static_cast<int64_t>(t.mt) * (2 * kTileM) + w.row_in_tile();
    if (t.first) acc = -INFINITY;
    ck.start();
    w.wait_full(it);
    ck.lap(ck.wait);
    if (epi_tid == 0 && it < 4) stamp(p, 4 + it);  // accumulator of sub-tile `it` ready
    const uint32_t taddr = w.taddr(buf);
    // one chunk per iteration, as when the ceiling in DESIGN.md was measured
#pragma unroll 1
    for (int c0 = 0; c0 < t.nvalid; c0 += kChunk) {
      uint32_t r[kChunk];
      ck.start();
      ptx::tmem_ld_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      ck.lap(ck.ld);
#pragma unroll
      for (int j = 0; j < kChunk; ++j) acc = fmaxf(acc, __uint_as_float(r[j]));
    }
    w.release(buf);
    if (epi_tid == 0 && it < 2) stamp(p, 14 + it);  // buffer of sub-tile `it` handed back
    if (epi_tid == 0 && it < 4) stamp(p, 8 + it);   // this warp is done with sub-tile `it`
    if (t.last && row < p.B) {
      const int64_t li = list_offset(p, w.pair, t.mt, row);
      p.part_val[li] = acc;
      p.part_idx[li] = -1;
    }
    ++it;
  }
  epi_done(p, ck, epi_tid);
}

// ===================== epilogue: deferred-insert top-K lists (production; umma_common.cuh) =====================
// A sorted register list per row.  Every sub-tile is filtered against a threshold fixed for the sub-tile into the
// thread's candidate queue; the queue is drained into the list once the accumulator buffer is back with the tensor core.
// kGroups: on the grouped schedule -- only the walk and the list slot differ.
template <int KL, bool kGroups>
__device__ __forceinline__ void epi_topk_defer(const Params& p, const EpiWarp& w, float* staging) {
  const int epi_tid = w.epi_tid();
  auto walk = WalkerOf<kGroups>::make(p, w.pair);
  SubTile t;
  SortedList<KL> list;
  list.init();
  float floor_thr = -INFINITY;   // warm-up floor of the segment
  CandQueue<defer_queue_len<KL>()> cq;
  cq.init(ptx::smem_u32(reinterpret_cast<uint2*>(staging) + epi_tid));
#ifdef HGR_PLACEMENT
  unsigned long long n_chunks = 0, n_crowded = 0;
#endif
  int it = 0;
  EpiClock ck(p.timeline != nullptr && epi_tid == 0);
  while (walk.next(t)) {
    const int buf = it & 1;
    const int64_t row = static_cast<int64_t>(t.mt) * (2 * kTileM) + w.row_in_tile();
    if (t.first) list.init();
    ck.start();
    w.wait_full(it);
    ck.lap(ck.wait);
    if (epi_tid == 0 && it < 4) stamp(p, 4 + it);  // accumulator of sub-tile `it` ready
    const uint32_t taddr = w.taddr(buf);
    if (t.first) floor_thr = warmup_floor_pairs<KL>(taddr, t.nvalid);
    ck.lap(ck.warm);
    float sub_thr = fmaxf(floor_thr, list.thr());   // fixed for the whole sub-tile
    for (int c0 = 0; c0 < t.nvalid; c0 += kChunk) {
      uint32_t r[kChunk];
      ck.start();
      ptx::tmem_ld_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      ck.lap(ck.ld);
      const int nv = t.nvalid - c0;
      const bool roomy = __reduce_max_sync(0xffffffffu, cq.count()) <= cq.kEntries - kChunk;
#ifdef HGR_PLACEMENT
      ++n_chunks;
      n_crowded += roomy ? 0 : 1;
#endif
      // Long lists (many survivors per sub-tile) make room up front; short lists rarely pass half of the queue, and
      // when a lane does they take the saturating append below, so that only a queue that really fills up makes the
      // warp drain while it still holds the TMEM buffer (measured: KL = 8 -0.2 us, KL = 16 +7 us with the lazy rule).
      if (!roomy && KL > 10) {
        ck.lap(ck.scan);
        cand_drain<KL>(list, cq);
        sub_thr = fmaxf(sub_thr, list.thr());
        ck.lap(ck.drain);
      }
      if (roomy || KL > 10) {
        if (nv >= kChunk) cand_append_chunk_roomy<true>(cq, r, nv, t.col0 + c0, sub_thr);
        else cand_append_chunk_roomy<false>(cq, r, nv, t.col0 + c0, sub_thr);
        ck.lap(ck.scan);
        continue;
      }
      const uint32_t wr0 = cq.wr;
      if (!cand_append_chunk(cq, r, nv, t.col0 + c0, sub_thr)) {  // a lane ran out of slots (rare):
        cq.wr = wr0;                                              // rewind, insert what is queued,
        ck.lap(ck.scan);
        cand_drain<KL>(list, cq);                                 // tighten the threshold and redo the chunk
        sub_thr = fmaxf(sub_thr, list.thr());
        ck.lap(ck.drain);
        if (!cand_append_chunk(cq, r, nv, t.col0 + c0, sub_thr)) {
          // more survivors in ONE chunk than the queue holds (list still warming up): insert straight
          // from TMEM, column by column
          cq.wr = cq.base;
          scan_chunk_reload<KL>(list, r, nv, taddr + c0, t.col0 + c0);
          sub_thr = fmaxf(sub_thr, list.thr());
        }
      }
      ck.lap(ck.scan);
    }
    w.release(buf);
    if (epi_tid == 0 && it < 2) stamp(p, 14 + it);  // buffer of sub-tile `it` handed back
    ck.start();                                     // the tensor core has the buffer: now pay for the inserts
    cand_drain<KL>(list, cq);
    ck.lap(ck.drain);
    if (epi_tid == 0 && it < 4) stamp(p, 8 + it);   // this warp is done with sub-tile `it`
    if (t.last && row < p.B) {
      int64_t li;
      if constexpr (kGroups)
        li = (static_cast<int64_t>(group_slot(p.sched, p.groups, t.mt, walk.unit_of(t), t.group)) * p.B + row) * p.KL;
      else
        li = list_offset(p, w.pair, t.mt, row);
      float* pv = p.part_val + li;
      int32_t* pi = p.part_idx + li;
#pragma unroll
      for (int k = 0; k < KL; ++k) {
        if (k < p.KL) {
          pv[k] = list.v[k];
          pi[k] = list.i[k];
        }
      }
    }
    ++it;
  }
  epi_done(p, ck, epi_tid);
#ifdef HGR_PLACEMENT
  if (w.lane == 0) place::count_chunks(n_chunks, n_crowded);
#endif
}

// ===================== epilogue: floor sketch + candidate queue (sketch_epi.cuh) =====================
__device__ __forceinline__ void epi_sketch(const Params& p, const EpiWarp& w, float* staging) {
  const int epi_tid = w.epi_tid();
  const uint32_t epoch = p.stats[1] + 1u;   // stays put until the last CTA of this launch has finished
  TileWalker walk(p.sched, w.pair, p.C);
  SubTile t;
  Sketch sk;
  FloorSlots fs;
  SkQueue q;
  q.init(ptx::smem_u32(reinterpret_cast<uint2*>(staging) + epi_tid));
  sk.init();
  fs.init(nullptr, epoch, 0);
  SkFloor floor;
  floor.init();
  float floor_seen = -INFINITY;   // floor.keep at the last compaction
  int slot = 0;
  bool solo = true;
  int it = 0;
  EpiClock ck(p.timeline != nullptr && epi_tid == 0);
  SkProf prof;
  prof.on = ck.on;
  while (walk.next(t)) {
    const int buf = it & 1;
    const int64_t row = static_cast<int64_t>(t.mt) * (2 * kTileM) + w.row_in_tile();
    const bool row_ok = row < p.B;
    if (t.first) {
      sk.init();
      floor.init();
      floor_seen = -INFINITY;
      q.reset();
      slot = w.pair - p.sched.first_cta(t.mt);
      solo = p.sched.parts(t.mt) == 1;   // the only list of its rows: no global floor, its own sketch is all there is
      fs.init(row_ok ? p.sk_floors + row * kSkSlots : nullptr, epoch, slot);
    }
    ck.start();
    w.wait_full(it);
    ck.lap(ck.wait);
    if (epi_tid == 0 && it < 4) stamp(p, 4 + it);
    const uint32_t taddr = w.taddr(buf);
    const int phase = t.col0 & 16;       // chunk starts are multiples of 32 from the sub-tile's first column
    // The row's global floor words.  The workers of a row tile run in step: what the others published after their
    // previous sub-tile is in by the time this accumulator is complete.  Fetch at chunk `fetch_at`, consume a few
    // chunks further down (or at once when the queue is crowded), so that the L2 round trip hides behind the chunks
    // in between.
    // The words come in two halves (10 words = 20 registers in flight at a time): half 0 is fetched at chunk
    // `fetch_at`, folded two chunks later while half 1 goes out, and the floor rises another two chunks on.
    int fetch_at = 0;
    if (t.first) {
      // A list that starts empty would take everything: one extra pass over the sub-tile (TMEM is re-readable)
      // builds the sketch first, so that its own columns are already filtered against their floor.  The class
      // maxima are published at once -- every list of the row does this at about the same time, so a few chunks
      // into the filter pass the GLOBAL floor of the row's first sub-tiles is there and almost nothing passes.
      for (int c0 = 0; c0 + kChunk <= t.nvalid; c0 += kChunk) {
        uint32_t r[kChunk];
        ptx::tmem_ld_x32(taddr + c0, r);
        ptx::tmem_ld_wait();
        sk.update(r, phase);
      }
      floor.raise(sk.floor());
      if (!solo) fs.publish(sk);
      fetch_at = kChunk;
      ck.lap(ck.warm);
    }
    int stage = solo ? 3 : 0;      // 0: nothing out, 1: half 0 in flight, 2: half 1 in flight, 3: done
    ck.start();
    const long long t_scan0 = ck.on ? clock64() : 0;
    for (int c0 = 0; c0 < t.nvalid; c0 += kChunk) {
      uint32_t r[kChunk];
      ptx::tmem_ld_x32(taddr + c0, r);
      if (stage == 0 && c0 >= fetch_at) {
        fs.fetch(0);
        stage = 1;
      } else if (stage == 1 && c0 >= fetch_at + 2 * kChunk) {
        fs.take(true);
        fs.fetch(1);
        stage = 2;
      } else if (stage == 2 && c0 >= fetch_at + 4 * kChunk) {
        fs.take(false);
        floor.raise(fs.floor());
        stage = 3;
      }
      ptx::tmem_ld_wait();
      const int nv = t.nvalid - c0;
      if (!t.first && solo && nv >= kChunk) {
        sk.update(r, phase);
        floor.raise(sk.floor());
      }
      sk_filter_chunk(q, r, nv, t.col0 + c0, floor, floor_seen, p.stats, &prof);
    }
    ck.lap(ck.scan);
    if (ck.on && blockIdx.x < 256 && t.seq < 3) p.timeline[blockIdx.x * kTimelineSlots + 24 + t.seq] = clock64() - t_scan0;
    w.release(buf);
    ck.start();
    // a short sub-tile: finish the fetch sequence now (the buffer is already back with the tensor core)
    if (stage == 1) {
      fs.take(true);
      fs.fetch(1);
      stage = 2;
    }
    if (stage == 2) {
      fs.take(false);
      floor.raise(fs.floor());
    }
    if (t.first) q.pub = q.wr;                                  // covered by the class maxima published above
    else if (!t.last && !solo) sk_publish_new(q, fs, floor.keep);
    if (epi_tid == 0 && it < 4) stamp(p, 8 + it);
    if (t.last) {
      // the queue becomes the list: at most kSkCap entries, everything else is provably outside the row's top-K
      sk_compact(q, floor.keep);
      if (__any_sync(0xffffffffu, q.count() > kSkCap)) sk_select(q, floor, kSkCap, p.stats);
      const int cnt = q.count();
      const int maxc = __reduce_max_sync(0xffffffffu, cnt);
      const int64_t li = static_cast<int64_t>(slot) * p.B + (row_ok ? row : 0);
      if (row_ok) p.sk_cnt[li] = cnt;
      uint2* out = p.sk_part + li * kSkCap;
      uint32_t rd = q.base;
      for (int e0 = 0; e0 < maxc; e0 += 4, rd += 4 * kSkStride) {
        uint32_t xb[4], col[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) ptx::ld_shared_v2(rd + i * kSkStride, xb[i], col[i]);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (row_ok && e0 + i < cnt) out[e0 + i] = make_uint2(xb[i], col[i]);
      }
    }
    ck.lap(ck.drain);
    ++it;
  }
  epi_done(p, ck, epi_tid);
  if (ck.on && blockIdx.x < 256) {
    unsigned long long* tl = p.timeline + blockIdx.x * kTimelineSlots;
    tl[27] = prof.sel, tl[28] = prof.cmp, tl[29] = prof.crowded, tl[30] = prof.passes, tl[31] = prof.selects;
  }
}

// ===================== epilogue: per-level arg-max (row f1, main.py:163-176 without the [B, N] matrix) ==========
// thread = image row; the bank rows are sorted by level, so the level of a column is warp-uniform and changes a
// handful of times per worker: a running (max, first column) per row, flushed with ONE 64-bit atomicMax of the
// winner word (topk_list.cuh) per level.
__device__ __forceinline__ void epi_level(const Params& p, const EpiWarp& w) {
  TileWalker walk(p.sched, w.pair, p.C);
  SubTile t;
  int it = 0;
  int lvl = 0;
  float best = -INFINITY;
  int bcol = 0x7FFFFFFF;
  while (walk.next(t)) {
    const int buf = it & 1;
    const int64_t row = static_cast<int64_t>(t.mt) * (2 * kTileM) + w.row_in_tile();
    auto flush = [&]() {
      if (row < p.B && bcol != 0x7FFFFFFF)
        atomicMax(p.lvl_best + row * p.n_levels + lvl, winner_word(order_key(best), static_cast<uint32_t>(bcol)));
      best = -INFINITY;
      bcol = 0x7FFFFFFF;
    };
    if (t.first) {
      lvl = 0;
      while (lvl < p.n_levels - 1 && t.col0 >= p.lvl_end[lvl]) ++lvl;
      best = -INFINITY;
      bcol = 0x7FFFFFFF;
    }
    w.wait_full(it);
    const uint32_t taddr = w.taddr(buf);
    for (int c0 = 0; c0 < t.nvalid; c0 += kChunk) {
      uint32_t r[kChunk];
      ptx::tmem_ld_x32(taddr + c0, r);
      ptx::tmem_ld_wait();
      const int cbeg = t.col0 + c0;
      const int nv = t.nvalid - c0 < kChunk ? t.nvalid - c0 : kChunk;
      if (cbeg + nv <= p.lvl_end[lvl] || lvl == p.n_levels - 1) {   // the whole chunk lies in the current level
        // four interleaved running maxima (a single one is a 32-deep chain of dependent compare + select pairs),
        // folded by (value desc, column asc) -- `>` keeps the first of equal values inside a stream
        float b4[4] = {best, -INFINITY, -INFINITY, -INFINITY};
        int c4[4] = {bcol, 0x7FFFFFFF, 0x7FFFFFFF, 0x7FFFFFFF};
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
          const float x = __uint_as_float(r[j]);
          if (j < nv && x > b4[j & 3]) {
            b4[j & 3] = x;
            c4[j & 3] = cbeg + j;
          }
        }
        best = b4[0];
        bcol = c4[0];
#pragma unroll
        for (int q = 1; q < 4; ++q) {
          if (b4[q] > best || (b4[q] == best && c4[q] < bcol)) {
            best = b4[q];
            bcol = c4[q];
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
          if (j < nv) {
            while (lvl < p.n_levels - 1 && cbeg + j >= p.lvl_end[lvl]) {
              flush();
              ++lvl;
            }
            const float x = __uint_as_float(r[j]);
            if (x > best) {
              best = x;
              bcol = cbeg + j;
            }
          }
        }
      }
    }
    w.release(buf);
    if (t.last) flush();
    ++it;
  }
}

template <int EPI, int KL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(EpiRes<EPI>::kThreads, 1)
score_umma_pair_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_bank,
                       const Params p) {
  HGR_PLACE_ENTER();
  using R = EpiRes<EPI, KL>;
  const int stages = p.stages;   // <= R::kMaxStages, chosen by the launcher (EpiRes::stages)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* staging = reinterpret_cast<float*>(smem + stages * kPairStageBytes);
  PairCtl* ctl = reinterpret_cast<PairCtl*>(smem + stages * kPairStageBytes + R::kStagingBytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();  // 0 = leader (issues the MMAs), 1 = peer
  const int pair = blockIdx.x >> 1;

  if (blockIdx.x == 0 && threadIdx.x == 0 && p.stats != nullptr) p.stats[0] = 0;
  if (threadIdx.x == 0) stamp(p, 0);  // kernel entry
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_bank);
    for (int s = 0; s < stages; ++s) {
      ptx::mbar_init(&ctl->full[s], 1);
      ptx::mbar_init(&ctl->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&ctl->tmem_full[b], 1);
      ptx::mbar_init(&ctl->tmem_empty[b], R::kTmemEmptyArrivals);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_cg2(&ctl->tmem_base, kTmemCols);
    ptx::tmem_relinquish_cg2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // barriers of both CTAs initialised, TMEM allocated
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctl->tmem_base;
  if (threadIdx.x == 0) stamp(p, 1);  // set-up done (barriers, TMEM, cluster sync)

  constexpr bool kGroups = EPI == kEpiTopkGroups;
  if (warp == 0) {
    produce<kGroups>(&map_x, &map_bank, p, ctl, smem, rank, pair);
  } else if (warp == 1) {
    if (rank == 0) issue_mma<kGroups>(p, ctl, smem, tmem_base, pair, lane);   // the leader's MMAs cover both CTAs
  } else {
    const EpiWarp w{ctl, tmem_base, rank, pair, warp, lane};
    if constexpr (EPI == kEpiDense) epi_dense(p, w, staging);
    else if constexpr (EPI == kEpiNull) epi_null(p, w);
    else if constexpr (EPI == kEpiTopkDefer) epi_topk_defer<KL, false>(p, w, staging);
    else if constexpr (EPI == kEpiTopkGroups) epi_topk_defer<KL, true>(p, w, staging);
    else if constexpr (EPI == kEpiSketch) epi_sketch(p, w, staging);
    else epi_level(p, w);
  }

  // no CTA may exit (or free TMEM) while its partner can still signal its barriers or read its memory
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_cg2(tmem_base, kTmemCols);
  }
  if (threadIdx.x == 32) stamp(p, 13);  // exit
  if (EPI == kEpiSketch && threadIdx.x == 0) {
    // the last CTA to finish advances the workspace's epoch: the next launch starts with empty floor words
    __threadfence();
    if (atomicAdd(&p.stats[2], 1u) == gridDim.x - 1) {
      p.stats[2] = 0;
      __threadfence();
      atomicAdd(&p.stats[1], 1u);
    }
  }
  HGR_PLACE_LEAVE(kScore);
}

template <int EPI, int KL>
int launch_one(const CUtensorMap& mx, const CUtensorMap& mb, const Params& p, cudaStream_t stream) {
  using R = EpiRes<EPI, KL>;
  Params pp = p;
  pp.stages = R::stages(p.B);
  auto kern = score_umma_pair_kernel<EPI, KL>;
  // the opt-in limit is a per-function attribute: always ask for the deepest ring so that concurrent callers with
  // different stage counts cannot lower it under each other
  HGR_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(R::smem_bytes(R::kMaxStages))));
  kern<<<2 * p.sched.G, R::kThreads, R::smem_bytes(pp.stages), stream>>>(mx, mb, pp);
  HGR_CHECK_LAUNCH();
  return HGR_OK;
}

}  // namespace

#ifdef HGR_PLACEMENT
// Diagnostics builds only: log into `rec` (cap records, `n` counts them) and `chunks` from now on; null pointers stop.
extern "C" int hgr_placement_attach(void* rec, void* n, unsigned int cap, void* chunks) {
  const place::Log l{static_cast<place::Rec*>(rec), static_cast<unsigned int*>(n), cap,
                     static_cast<unsigned long long*>(chunks)};
  int rc = place::attach(l);
  if (rc == HGR_OK) rc = placement_attach_normalize(l);
  return rc == HGR_OK ? placement_attach_merge(l) : rc;
}
#endif

int pair_ring_depth(int64_t B) { return EpiRes<kEpiTopkDefer>::stages(B); }

template <int KL>
int footprint_one(int64_t B, int32_t* out) {
  using R = EpiRes<kEpiTopkDefer, KL>;
  cudaFuncAttributes fa;
  HGR_CHECK_CUDA(cudaFuncGetAttributes(&fa, score_umma_pair_kernel<kEpiTopkDefer, KL>));
  out[0] = R::kThreads;
  out[1] = fa.numRegs;
  out[2] = static_cast<int32_t>(fa.sharedSizeBytes);
  out[3] = static_cast<int32_t>(R::smem_bytes(R::stages(B)));   // what launch_one asks for
  return HGR_OK;
}

int pair_kernel_footprint(int64_t B, int KL, int32_t* out) {
  switch (KL) {
    case 8: return footprint_one<8>(B, out);
    case 10: return footprint_one<10>(B, out);
    case 12: return footprint_one<12>(B, out);
    case 16: return footprint_one<16>(B, out);
    case 20: return footprint_one<20>(B, out);
    case 32: return footprint_one<32>(B, out);
  }
  return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk_footprint: list length %d", KL);
}

template <int EPI>
int launch_topk(int KL, const CUtensorMap& mx, const CUtensorMap& mb, const Params& p, cudaStream_t stream) {
  switch (KL) {
    case 8: return launch_one<EPI, 8>(mx, mb, p, stream);
    case 10: return launch_one<EPI, 10>(mx, mb, p, stream);
    case 12: return launch_one<EPI, 12>(mx, mb, p, stream);
    case 16: return launch_one<EPI, 16>(mx, mb, p, stream);
    case 20: return launch_one<EPI, 20>(mx, mb, p, stream);
    case 32: return launch_one<EPI, 32>(mx, mb, p, stream);
  }
  return set_error(HGR_ERR_UNSUPPORTED, "hgr_score_topk(tcgen05): list length %d", KL);
}

// Epilogue arrangement of the top-K kernels: ONE warp per TMEM lane quarter, one list per row, inserts deferred off the
// tensor core's critical path (measured against two warps per quarter with in-place inserts: exact 20-entry lists at
// B = 4096 40 / 57 / 87 / 154 us against 46 / 66 / 98 / 164 us).  The dense epilogue uses two warps per quarter.
int launch_pair_kernel(int epi, int KL, const CUtensorMap& mx, const CUtensorMap& mb, const Params& p,
                       cudaStream_t stream) {
  if (epi == kEpiDense) return launch_one<kEpiDense, 8>(mx, mb, p, stream);
  if (epi == kEpiNull) return launch_one<kEpiNull, 8>(mx, mb, p, stream);
  if (epi == kEpiSketch) return launch_one<kEpiSketch, 8>(mx, mb, p, stream);
  if (epi == kEpiLevel) return launch_one<kEpiLevel, 8>(mx, mb, p, stream);
  if (epi == kEpiTopkGroups) return launch_topk<kEpiTopkGroups>(KL, mx, mb, p, stream);
  return launch_topk<kEpiTopkDefer>(KL, mx, mb, p, stream);
}

}  // namespace umma
}  // namespace hgr
