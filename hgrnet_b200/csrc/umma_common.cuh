// Device-side pieces of the tcgen05 scoring kernel (score_pair.cu): kernel parameters and the deferred-insert top-K
// epilogue (sorted per-row lists).  The work split lives in sched.cuh, the floor-sketch epilogue in sketch_epi.cuh.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "ptx.cuh"
#include "topk_list.cuh"

namespace hgr {
namespace umma {

constexpr int kBlockK = 64;                         // bf16 per K block: 128 bytes = one swizzle row
constexpr int kUmmaK = 16;                          // K of one tcgen05.mma.kind::f16
constexpr int kABytes = kTileM * kBlockK * 2;       // 16 KB
constexpr int kBBoxRows = 64;                       // bank rows per TMA box
constexpr int kBBoxBytes = kBBoxRows * kBlockK * 2; // 8 KB
constexpr int kEpiWarp0 = 2;
constexpr int kTmemCols = 512;
constexpr int kChunk = 32;                          // accumulator columns per tcgen05.ld
constexpr int kMaxHierLevels = 32;                  // hierarchy levels of the per-level arg-max epilogue

// kEpiTopkGroups: the kEpiTopkDefer epilogue on the grouped schedule (Params::groups, hgr_score_topk_splits)
enum EpiMode { kEpiDense = 0, kEpiNull = 3, kEpiTopkDefer = 4, kEpiSketch = 5, kEpiLevel = 6, kEpiTopkGroups = 7 };
enum Variant { kVarProd = 0, kVarExact = 2, kVarNull = 3, kVarSketch = 10 };   // impl code - HGR_IMPL_TCGEN05

// SubTile / TileWalker (the walk of one worker over its chunk of the schedule) live in sched.cuh: plain integer
// arithmetic, shared with the host-side unit test of the schedule (tests/test_cpu_sched.py).
using ::hgr::SubTile;
using ::hgr::TileWalker;

struct Params {
  Sched sched;
  int64_t B, C;
  int num_k_blocks;
  int KL;              // entries written per list
  float scale;
  float* part_val;     // [slots][B][KL]
  int32_t* part_idx;   // [slots][B][KL] bank rows
  float* dense_out;    // [B][ldo]
  int64_t ldo;
  unsigned int* stats; // [0] = rows re-scanned by the merge kernel of this call (reset here)
  unsigned long long* timeline;  // optional [CTA][24] %globaltimer stamps (HGR_TIMELINE=1), else nullptr
  int stages;          // operand ring depth of the CTA-pair kernel (set by its launcher)
  // floor-sketch epilogue (sketch_epi.cuh); stats[1] = launch epoch of the workspace, stats[2] = finished CTAs
  // per-level arg-max epilogue (kEpiLevel, row f1: TOR / POR without the dense logits): the bank rows are sorted by
  // hierarchy level, level l = rows [lvl_end[l-1], lvl_end[l]); lvl_best[row * n_levels + l] takes the in-level maximum
  // of a row as (order key << 32 | ~bank row) by atomicMax (0 = no column seen; the finishing kernel zeroes what it reads)
  int n_levels;
  int lvl_end[kMaxHierLevels];
  unsigned long long* lvl_best;
  uint2* sk_part;                  // [slots][B][kSkCap] (value bits, bank row)
  int32_t* sk_cnt;                 // [slots][B] entries of each list
  unsigned long long* sk_floors;   // [B][kSkSlots] (epoch << 32 | order key)
  // grouped schedule (kEpiTopkGroups): no list holds rows of two groups, list slots per group_slot (sched.cuh)
  Groups groups;
};

constexpr int kTimelineSlots = 32;
constexpr int kWsHeaderBytes = kScoreWsHeaderBytes;  // statistics + timeline stamps in front of the partial lists
static_assert(kWsHeaderBytes >= 64 + 256 * kTimelineSlots * 8, "the header holds the statistics and the timeline stamps");

__device__ __forceinline__ void stamp(const Params& p, int slot) {
  if (p.timeline != nullptr && blockIdx.x < 256) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.timeline[blockIdx.x * kTimelineSlots + slot] = t;
  }
}
// cycle accounting of one epilogue warp (profiling builds of the timeline only)
struct EpiClock {
  long long ld = 0, scan = 0, drain = 0, wait = 0, warm = 0;
  long long t = 0;
  bool on;
  __device__ __forceinline__ explicit EpiClock(bool enable) : on(enable) {}
  __device__ __forceinline__ void start() { if (on) t = clock64(); }
  __device__ __forceinline__ void lap(long long& acc) {
    if (on) {
      const long long n = clock64();
      acc += n - t;
      t = n;
    }
  }
};

template <int KL>
__device__ __forceinline__ void scan_chunk_reload(SortedList<KL>& list, const uint32_t (&r)[kChunk], int nv,
                                                  uint32_t taddr_chunk, int col_chunk) {
  const float thr = list.thr();
  uint32_t m = 0;
#pragma unroll
  for (int j = 0; j < kChunk; ++j)
    if (__uint_as_float(r[j]) > thr) m |= (1u << j);
  if (nv < kChunk) m &= (1u << nv) - 1u;
  uint32_t wm = __reduce_or_sync(0xffffffffu, m);
  // visit the union of positions in ascending order; each lane re-reads its own value of that
  // column from TMEM (the address is warp-uniform) and inserts if it still qualifies
  while (wm) {
    const int j = __ffs(wm) - 1;
    wm &= wm - 1;
    const float x = __uint_as_float(ptx::tmem_ld_x1(taddr_chunk + j));
    ptx::tmem_ld_wait();
    if (((m >> j) & 1u) && x > list.thr()) list.insert(x, col_chunk + j);
  }
}

// Warm-up floor of a segment.  A list that starts empty accepts everything, and the insert body is what the epilogue
// pays for (ALU pipe).  Before scanning the first sub-tile of a segment the warp therefore takes one cheap extra pass
// over that sub-tile (TMEM is re-readable): G = KL / 2 interleaved groups, each tracking its TWO largest values
// (3 FMNMX per value, no divergence).  tau = the smallest runner-up is reached by at least 2 * G = KL columns, i.e. it
// is a valid lower bound of the list's final KL-th entry, so everything below tau can be dropped up front without
// touching the certificate argument (dropped <= final last entry).  For KL = 8 over 256 columns ~14 values survive;
// the worst lane of a warp -- what the lock-step drain pays for -- ~26.  Full chunks only: a ragged tail chunk is
// simply left out (any subset of the stream gives a valid bound).  Returns the largest float below tau (ties with
// tau must still enter), or -inf when the sub-tile is too small to fill every group.
template <int KL>
__device__ __forceinline__ float warmup_floor_pairs(uint32_t taddr, int nvalid) {
  constexpr int G = KL / 2;
  static_assert(KL % 2 == 0 && G >= 1, "pair floor needs an even list length");
  if (nvalid < kChunk) return -INFINITY;
  float hi[G], lo[G];
#pragma unroll
  for (int g = 0; g < G; ++g) hi[g] = lo[g] = -INFINITY;
  for (int c0 = 0; c0 + kChunk <= nvalid; c0 += kChunk) {
    uint32_t r[kChunk];
    ptx::tmem_ld_x32(taddr + c0, r);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
      const float x = __uint_as_float(r[j]);
      lo[j % G] = fmaxf(lo[j % G], fminf(hi[j % G], x));
      hi[j % G] = fmaxf(hi[j % G], x);
    }
  }
  float tau = lo[0];
#pragma unroll
  for (int g = 1; g < G; ++g) tau = fminf(tau, lo[g]);
  return nextafterf(tau, -INFINITY);
}

// ---- deferred-insert epilogue -------------------------------------------------------------------------------
// The accumulator buffer is only needed while its values are FILTERED; the (ALU-bound) sorted inserts can run
// from shared memory afterwards.  So a sub-tile is scanned against a threshold that is fixed for the whole
// sub-tile (warm-up floor / the list's current KL-th value), survivors are appended as (value, column) pairs
// to a per-thread queue, the TMEM buffer is handed back to the MMA warp at once, and only then is the queue
// drained into the list -- in lock-step over one dense batch per sub-tile, while the tensor core already works
// two sub-tiles ahead.  The epilogue leaves the critical path of the MMAs entirely.
// Queue entries per thread (+1 dud slot) for lists of KL entries.  Narrow lists (KL <= 10) keep 56: the 8 KB this
// frees beside 5 operand stages let a normalise and two merge CTAs share the SM with a resident scoring CTA
// (DESIGN.md section 4, budget rule).  Measured at cfg 2 (tools/placement.py): 2.3 % of the chunks then find some
// lane's queue too full for the roomy append (0.13 % with 64 entries) and take the saturating one; the scoring kernel
// alone at full clock is unchanged (24.64 vs 24.69 us).  Wider lists keep 64.
template <int KL>
constexpr int defer_queue_len() { return KL <= 10 ? 56 : 64; }
constexpr uint32_t kDeferStride = 128 * 8;        // one entry of each of the CTA's 128 epilogue threads
template <int kLen>
struct CandQueue {
  static constexpr int kEntries = kLen;
  uint32_t base;  // shared-space byte address of entry 0 of this thread; entries are kDeferStride bytes apart
  uint32_t wr;    // next free entry
  __device__ __forceinline__ void init(uint32_t b) { base = wr = b; }
  __device__ __forceinline__ uint32_t limit() const { return base + kLen * kDeferStride; }  // the dud slot
  __device__ __forceinline__ int count() const { return static_cast<int>((wr - base) / kDeferStride); }
};

// Branch-free append: every value is stored at the write cursor, the cursor only advances for survivors (the
// next store overwrites a non-survivor) and saturates at the last slot, which therefore only ever holds duds.
// (Inline-asm stores inside an `if` would be compiled as 32 divergent branches per chunk.)  The queue has
// kLen + 1 entries per thread.  Returns false when some lane of the warp ran out of slots: the caller then
// rewinds, drains and appends the same chunk again.
template <int kLen>
__device__ __forceinline__ bool cand_append_chunk(CandQueue<kLen>& q, const uint32_t (&r)[kChunk], int nv,
                                                  int col_chunk, float thr) {
  uint32_t wr = q.wr;
  const uint32_t lim = q.limit();
#pragma unroll
  for (int j = 0; j < kChunk; ++j) {
    const bool pass = (__uint_as_float(r[j]) > thr) && (nv >= kChunk || j < nv);  // ragged tail: drop columns >= C
    ptx::st_shared_v2(wr, r[j], static_cast<uint32_t>(col_chunk + j));
    wr += pass ? kDeferStride : 0;
    wr = wr < lim ? wr : lim;
  }
  q.wr = wr;
  return !__any_sync(0xffffffffu, wr >= lim);
}

// Same without the per-value saturation (one op less on the cursor's dependency chain): the caller guarantees
// room for a whole chunk (count <= kLen - 32 in every lane).
template <bool FULL, int kLen>
__device__ __forceinline__ void cand_append_chunk_roomy(CandQueue<kLen>& q, const uint32_t (&r)[kChunk],
                                                        int nv, int col_chunk, float thr) {
  uint32_t wr = q.wr;
  // store-all / advance-on-pass: every value is written at the cursor and the next store overwrites a
  // non-survivor.  (Predicating the store and the bump in PTX instead -- no write for a non-survivor -- measured
  // 70 % SLOWER: the store's address then hangs on a 2-instruction predicated chain per value.)
#pragma unroll
  for (int j = 0; j < kChunk; ++j) {
    const bool pass = (__uint_as_float(r[j]) > thr) && (FULL || j < nv);
    ptx::st_shared_v2(wr, r[j], static_cast<uint32_t>(col_chunk + j));
    wr += pass ? kDeferStride : 0;
  }
  q.wr = wr;
}

template <int KL, int kLen>
__device__ __forceinline__ void cand_drain(SortedList<KL>& list, CandQueue<kLen>& q) {
  const int cnt = q.count();
  const int maxc = __reduce_max_sync(0xffffffffu, cnt);
  uint32_t rd = q.base;
  // the next entry is fetched while the current one is inserted (one warp per scheduler: nothing else would hide
  // the shared-memory latency); reading one entry past a lane's count stays inside its kLen + 1 slots
  uint32_t xb, col;
  ptx::ld_shared_v2(rd, xb, col);
  for (int e = 0; e < maxc; ++e) {
    const float x = e < cnt ? __uint_as_float(xb) : -INFINITY;
    const int32_t c = static_cast<int32_t>(col);
    rd += kDeferStride;
    ptx::ld_shared_v2(rd, xb, col);
    if (x > list.thr()) list.insert(x, c);
  }
  q.wr = q.base;
}

// score_pair.cu
int pair_ring_depth(int64_t B);   // operand stages of the production (deferred-insert) kernel for a batch size
// {threads, registers per thread, static shared memory, dynamic shared memory} of the production kernel as
// launch_pair_kernel launches it for B rows and lists of KL entries
int pair_kernel_footprint(int64_t B, int KL, int32_t* out);
int launch_pair_kernel(int epi, int KL, const CUtensorMap& mx, const CUtensorMap& mb, const Params& p,
                       cudaStream_t stream);

}  // namespace umma
}  // namespace hgr
