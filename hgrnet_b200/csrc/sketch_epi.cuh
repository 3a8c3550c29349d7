// Fused top-K epilogue of the tcgen05 scoring kernels: FLOOR SKETCH + CANDIDATE QUEUE (no sorted lists).
//
// Reference: `logits[:, test_index]` + `.topk(20, 1, True, True)` (main.py:136-138).  The reference materialises
// the B x C logits and sorts; here a thread (= one image row = one TMEM lane) sees its row's logits stream by, 32
// accumulator columns at a time, and has to hand the merge kernel every column that can be in the row's top-K.
//
// What a row keeps:
//  * a SKETCH of its first sub-tile: kSkGroups = 10 column classes (class of bank row c = (c & 31) % 10), each with its
//    two largest values (3 FMNMX per value).  The smallest runner-up tau is reached by >= 20 distinct columns, so
//    nothing below tau can be among the row's top-20: `floor` = the largest float below tau is a valid filter.  No
//    data-dependent control flow, no sorted insert.  (A list that is the ONLY one of its rows keeps sketching.)
//  * a share in the row's GLOBAL floor: the row's columns are streamed by several workers at once (one list per
//    worker and row).  Every worker publishes its class maxima into kSkSlots = 20 words per row in global memory
//    (`red.max`; class g of list l -> word 2 g + (l & 1), so distinct words hold distinct columns) and reads the 20
//    words back once per sub-tile: their minimum is a valid floor for the whole row -- it reflects every column any
//    worker has seen so far, not just this list's.  After the first sub-tile almost nothing passes the filter, however
//    many lists a row is split into and whatever order the bank rows come in (no speculation, no certificate, no
//    repair pass: the result is exact by construction).  Later on only SURVIVORS are published (from the queue, at
//    the end of a sub-tile): a value at or below the floor cannot raise a word, every word being >= their minimum.
//    Words carry the launch's epoch in their upper half, so a workspace never has to be cleared between launches.
//  * a QUEUE of (value, bank row) candidates in shared memory: the columns that passed the filter, in stream order
//    (branch-free store-all append).  When it is crowded it is re-filtered against the (risen) floor; if that does
//    not make room, an exact selection (bisection on order-preserving integer keys held in registers, ties by
//    ascending column) cuts it down to 20..24 entries and raises the row's private floor.  At the end of a segment
//    the queue (<= kSkCap entries) IS the list; topk_merge_counts_kernel selects the row's top-K from its lists.
// Status: exact on every bank order (tests/test_gpu_kernels.py::test_hostile_bank_orders) but slower than the
// deferred-insert lists on shuffled banks -- not the production path; measurements in profiles/r02_sketch_experiments.md.
#pragma once
#include "umma_common.cuh"

namespace hgr {
namespace umma {

constexpr int kSkGroups = 10;   // column classes of the local sketch (top-2 each -> 20 witnesses)
constexpr int kSkSlots = 20;    // global floor words per image row
constexpr int kSkKeep = 20;     // witnesses behind every floor = the largest K the kernel serves
constexpr int kSkQueue = 64;    // queue entries per row
constexpr int kSkCap = 32;      // entries of a finished list; kSkQueue - kSkCap >= 32 = one chunk always fits
constexpr int kSkSelectTo = 24; // a mid-stream selection leaves 20..24 entries
constexpr int kSkThreads = 128; // epilogue threads per CTA (queue entries of one thread are kSkThreads * 8 bytes apart)
constexpr uint32_t kSkStride = kSkThreads * 8;
constexpr int kSkQueueBytes = (kSkQueue + 1) * kSkThreads * 8;   // + one dud slot per row (branch-free appends)
constexpr uint32_t kKeyNegInf = 0x007FFFFFu;   // order key (topk_list.cuh) of -inf; smaller keys are (negative) NaN patterns

// Filter threshold for "key(x) >= k": the largest float below the value of key k (x > result).  -inf when k is not
// above -inf.  A result of +-0 is replaced by the smallest negative float: the float compare treats -0 == +0, which
// would otherwise drop a +0 that the key order keeps (looser is always valid).
__device__ __forceinline__ float below_key(uint32_t k) {
  if (k <= kKeyNegInf) return -INFINITY;
  const float f = order_key_value(k - 1);
  return f == 0.0f ? __uint_as_float(0x80000001u) : f;
}
__device__ __forceinline__ float below(float tau) { return below_key(order_key(tau)); }

// Column classes are a function of the ABSOLUTE bank row: class(col) = (col & 31) % 10, so that the warm-up pass (which
// sees whole chunks) and the per-entry publishing (which sees single columns) agree.  A chunk starts at a multiple of
// 16: PH = chunk start & 31 is 0 or 16 and register j of the chunk holds column class ((j + PH) & 31) % 10.
__host__ __device__ constexpr int sk_class(int col) { return (col & 31) % kSkGroups; }

struct Sketch {
  float hi[kSkGroups], lo[kSkGroups];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int g = 0; g < kSkGroups; ++g) hi[g] = lo[g] = -INFINITY;
  }
  template <int PH>
  __device__ __forceinline__ void update_ph(const uint32_t (&r)[kChunk]) {
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
      const float x = __uint_as_float(r[j]);
      lo[sk_class(j + PH)] = fmaxf(lo[sk_class(j + PH)], fminf(hi[sk_class(j + PH)], x));
      hi[sk_class(j + PH)] = fmaxf(hi[sk_class(j + PH)], x);
    }
  }
  __device__ __forceinline__ void update(const uint32_t (&r)[kChunk], int phase) {
    if (phase) update_ph<16>(r);
    else update_ph<0>(r);
  }
  __device__ __forceinline__ float floor() const {   // valid filter threshold from this list's own columns
    float tau = lo[0];
#pragma unroll
    for (int g = 1; g < kSkGroups; ++g) tau = fminf(tau, lo[g]);
    return below(tau);
  }
};

// The row's share of the global floor: 20 x (epoch << 32 | key) words.
struct FloorSlots {
  unsigned long long* row;   // this row's slots (nullptr: row >= B, nothing is read or published)
  uint32_t epoch;
  int par;                   // slot of class g = 2 g + par
  unsigned long long v[kSkSlots / 2];   // one HALF of the words in flight at a time (register budget)
  uint32_t kmin;

  __device__ __forceinline__ void init(unsigned long long* row_slots, uint32_t epoch_, int list) {
    row = row_slots;
    epoch = epoch_;
    par = list & 1;
  }
  // issue the loads of half h (0 / 1) of the row's words; their latency hides behind the chunks processed before
  // the matching take()
  __device__ __forceinline__ void fetch(int h) {
    if (row == nullptr) return;
#pragma unroll
    for (int i = 0; i < kSkSlots / 4; ++i)
      asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(v[2 * i]), "=l"(v[2 * i + 1]) : "l"(row + h * (kSkSlots / 2) + 2 * i) : "memory");
  }
  // fold the half fetched last into the running minimum (start == first half)
  __device__ __forceinline__ void take(bool start) {
    uint32_t m = start ? 0xFFFFFFFFu : kmin;
#pragma unroll
    for (int i = 0; i < kSkSlots / 2; ++i) {
      const uint32_t k = static_cast<uint32_t>(v[i] >> 32) == epoch ? static_cast<uint32_t>(v[i]) : 0u;
      m = k < m ? k : m;
    }
    kmin = m;
  }
  // floor of the whole row once both halves are in
  __device__ __forceinline__ float floor() const { return row == nullptr ? -INFINITY : below_key(kmin); }
  __device__ __forceinline__ void red_max(int cls, uint32_t key) const {
    const unsigned long long w = (static_cast<unsigned long long>(epoch) << 32) | key;
    asm volatile("red.relaxed.gpu.global.max.u64 [%0], %1;" ::"l"(row + 2 * cls + par), "l"(w) : "memory");
  }
  // all class maxima of a fresh sketch (first sub-tile of a segment)
  __device__ __forceinline__ void publish(const Sketch& sk) const {
    if (row == nullptr) return;
#pragma unroll
    for (int g = 0; g < kSkGroups; ++g) {
      const uint32_t k = order_key(sk.hi[g]);
      if (k > kKeyNegInf) red_max(g, k);
    }
  }
};

// The filter threshold of a row.  `in` filters NEW columns (x > in passes), `keep` re-filters the queue (x > keep
// stays).  They differ only after a tie cut (sk_select): the kept entries EQUAL the cut value and must survive later
// compactions, while every later column of that value loses the tie (larger column) and must not enter.
struct SkFloor {
  float in, keep;
  __device__ __forceinline__ void init() { in = keep = -INFINITY; }
  __device__ __forceinline__ void raise(float f) {
    in = fmaxf(in, f);
    keep = fmaxf(keep, f);
  }
};

struct SkQueue {
  uint32_t base, wr;   // shared-space byte addresses: entry 0 of this thread, next free entry
  uint32_t pub;        // first entry not yet published into the row's global floor words (base <= pub <= wr)
  __device__ __forceinline__ void init(uint32_t b) { base = wr = pub = b; }
  __device__ __forceinline__ void reset() { wr = pub = base; }
  __device__ __forceinline__ int count() const { return static_cast<int>((wr - base) / kSkStride); }
};

// Branch-free append of a chunk: EVERY value is stored at the cursor, the cursor only advances for survivors (the next
// store overwrites a non-survivor) -- straight-line code, which is what a lone warp per scheduler needs: nothing else
// would hide the latency of a data-dependent loop over the survivors (measured: ~150 cycles per survivor that way).
// The queue has kSkQueue + 1 slots, so the cursor may rest on slot kSkQueue (duds only).
// Pre-condition of the roomy form: count <= kSkQueue - kChunk in every lane.
template <bool FULL, int J0 = 0, int J1 = kChunk>
__device__ __forceinline__ void sk_append_roomy(SkQueue& q, const uint32_t (&r)[kChunk], int nv, int col_chunk, float floor) {
  uint32_t wr = q.wr;
#pragma unroll
  for (int j = J0; j < J1; ++j) {
    const bool pass = (__uint_as_float(r[j]) > floor) && (FULL || j < nv);   // ragged tail: columns >= C are zero fill
    ptx::st_shared_v2(wr, r[j], static_cast<uint32_t>(col_chunk + j));
    wr += pass ? kSkStride : 0u;
  }
  q.wr = wr;
}
// Saturating form for a crowded queue: false when some lane may have lost a survivor (the caller rewinds and redoes
// the chunk after making room).
__device__ __forceinline__ bool sk_append_sat(SkQueue& q, const uint32_t (&r)[kChunk], int nv, int col_chunk, float floor) {
  uint32_t wr = q.wr;
  const uint32_t lim = q.base + kSkQueue * kSkStride;
#pragma unroll
  for (int j = 0; j < kChunk; ++j) {
    const bool pass = (__uint_as_float(r[j]) > floor) && j < nv;
    ptx::st_shared_v2(wr, r[j], static_cast<uint32_t>(col_chunk + j));
    wr += pass ? kSkStride : 0u;
    wr = wr < lim ? wr : lim;
  }
  q.wr = wr;
  return !__any_sync(0xffffffffu, wr >= lim);
}

// Re-filter the queue against the floor, in place, keeping the stream order.  (One warp per scheduler: nothing hides
// a shared-memory round trip, so four entries are in flight per step.)  The published prefix stays a prefix.
__device__ __forceinline__ void sk_compact(SkQueue& q, float floor) {
  const int cnt = q.count();
  const int npub = static_cast<int>((q.pub - q.base) / kSkStride);
  const int maxc = __reduce_max_sync(0xffffffffu, cnt);
  uint32_t rd = q.base, w = q.base, wpub = q.base;
  for (int e0 = 0; e0 < maxc; e0 += 4) {
    uint32_t xb[4], col[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ptx::ld_shared_v2(rd + i * kSkStride, xb[i], col[i]);   // <= entry 63 (maxc <= 64)
    rd += 4 * kSkStride;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ptx::st_shared_v2(w, xb[i], col[i]);   // w <= the entry just read
      w += (e0 + i < cnt && __uint_as_float(xb[i]) > floor) ? kSkStride : 0u;
      wpub = e0 + i < npub ? w : wpub;
    }
  }
  q.wr = w;
  q.pub = wpub;
}

// New queue entries into the row's global floor words: entry (x, col) raises word 2 * class(col) + parity.  Only
// survivors are ever published -- a value at or below the row's floor cannot raise a word (every word is >= the floor,
// their minimum) -- and survivors are few, so no class maxima have to be tracked while filtering.
__device__ __forceinline__ void sk_publish_new(SkQueue& q, const FloorSlots& fs, float floor) {
  const int n = static_cast<int>((q.wr - q.pub) / kSkStride);
  const int maxn = __reduce_max_sync(0xffffffffu, n);
  uint32_t rd = q.pub;
  for (int e0 = 0; e0 < maxn; e0 += 2) {
    uint32_t xb[2], col[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      xb[i] = col[i] = 0;
      if (e0 + i < n) ptx::ld_shared_v2(rd + i * kSkStride, xb[i], col[i]);   // other lanes may have more new entries
    }
    rd += 2 * kSkStride;
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (e0 + i < n && fs.row != nullptr && __uint_as_float(xb[i]) > floor)
        fs.red_max(sk_class(static_cast<int>(col[i])), order_key(__uint_as_float(xb[i])));
  }
  q.pub = q.wr;
}

// Exact reduction of over-full queues (warp-uniform call; lanes with count <= limit keep everything).  For the
// others a key T is found by bisection with kSkKeep <= #{key >= T} <= limit; if ties make that impossible
// (#{key > T} < kSkKeep < limit < #{key >= T}), the kSkKeep - #{key > T} FIRST tied entries stay -- the queue is in
// ascending column order, so these are the ones the (value desc, column asc) order prefers, and every later column
// of that value loses the tie as well: the filter for new columns becomes the value of T itself (strict compare).
// The keys of all 64 slots are held in registers: a counting pass is 64 compare-and-add with four accumulators.
struct SkState {
  uint32_t wr, pub;
  float in, keep;
  int passes;
};
struct SkProf {   // cycle accounting of one epilogue warp (timeline builds only)
  long long sel = 0, cmp = 0;
  int crowded = 0, passes = 0, selects = 0;
  bool on = false;
};
static __device__ __noinline__ SkState sk_select_impl(uint32_t q_base, uint32_t q_wr, uint32_t q_pub, float f_in, float f_keep, int limit,
                                                     unsigned int* stat) {
  const int lane = threadIdx.x & 31;
  if (lane == 0 && stat != nullptr) atomicAdd(stat, 1u);
  const int cnt = static_cast<int>((q_wr - q_base) / kSkStride);
  const int maxc = __reduce_max_sync(0xffffffffu, cnt);
  const bool act = cnt > limit;
  uint32_t key[kSkQueue];
#pragma unroll
  for (int e = 0; e < kSkQueue; ++e) key[e] = order_key(ptx::ld_shared_f32(q_base + e * kSkStride));
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
#pragma unroll
  for (int e = 0; e < kSkQueue; ++e) {
    key[e] = e < cnt ? key[e] : 0u;          // empty slots never count (every real key is > 0)
    lo = (e < cnt && key[e] < lo) ? key[e] : lo;
    hi = key[e] > hi ? key[e] : hi;
  }
  int c_lo = cnt;   // #{key >= lo}
  int passes = 0;
  for (;;) {
    const bool go = act && lo < hi && c_lo > limit;
    if (!__any_sync(0xffffffffu, go)) break;
    ++passes;
    const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
    int c4[4] = {0, 0, 0, 0};
#pragma unroll
    for (int e = 0; e < kSkQueue; ++e) c4[e & 3] += key[e] >= mid ? 1 : 0;
    const int c = (c4[0] + c4[1]) + (c4[2] + c4[3]);
    if (go) {
      if (c >= kSkKeep) {
        lo = mid;
        c_lo = c;
      } else {
        hi = mid - 1u;
      }
    }
  }
  const bool ties = act && c_lo > limit;   // lo == hi: more than `limit` entries from the value of lo upwards
  int need = 0;
  if (ties) {
    int gt = 0;
#pragma unroll
    for (int e = 0; e < kSkQueue; ++e) gt += key[e] > lo ? 1 : 0;
    need = kSkKeep - gt;
  }
  // compaction, keeping the stream order (and the published prefix a prefix)
  const int npub = static_cast<int>((q_pub - q_base) / kSkStride);
  uint32_t rd = q_base, w = q_base, wpub = q_base;
  for (int e0 = 0; e0 < maxc; e0 += 4) {
    uint32_t xb[4], col[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ptx::ld_shared_v2(rd + i * kSkStride, xb[i], col[i]);
    rd += 4 * kSkStride;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ptx::st_shared_v2(w, xb[i], col[i]);
      const uint32_t k = order_key(__uint_as_float(xb[i]));
      bool keep = e0 + i < cnt;
      if (act) {
        const bool tied = k == lo;
        keep = keep && (k > lo || (tied && (!ties || need > 0)));
        need -= (ties && tied && e0 + i < cnt) ? 1 : 0;
      }
      w += keep ? kSkStride : 0u;
      wpub = e0 + i < npub ? w : wpub;
    }
  }
  SkState out;
  out.passes = passes;
  out.wr = w;
  out.pub = wpub;
  out.in = f_in;
  out.keep = f_keep;
  if (act) {
    const float f = below_key(lo);
    out.in = fmaxf(out.in, f);
    out.keep = fmaxf(out.keep, f);
    if (ties) out.in = fmaxf(out.in, order_key_value(lo));
  }
  return out;
}
// (by value in, by value out: references would pin the caller's cursor and floors in local memory)
__device__ __forceinline__ void sk_select(SkQueue& q, SkFloor& floor, int limit, unsigned int* stat, SkProf* prof = nullptr) {
  const long long t0 = (prof && prof->on) ? clock64() : 0;
  const SkState s = sk_select_impl(q.base, q.wr, q.pub, floor.in, floor.keep, limit, stat);
  if (prof && prof->on) {
    prof->sel += clock64() - t0;
    prof->passes += s.passes;
    prof->selects += 1;
  }
  q.wr = s.wr;
  q.pub = s.pub;
  floor.in = s.in;
  floor.keep = s.keep;
}

// Filter one chunk of 32 accumulator columns into the queue.  Straight-line code wherever possible: a lone warp per
// scheduler runs dependent, branchy code at a fraction of its issue rate (measured: a data-dependent loop over the
// survivors ~150 cycles per survivor, a chunk-maximum gate in front of the append +100 cycles per chunk, the branch-free
// store-all ~20 cycles per value).  A crowded queue (some lane above kSkQueue - kChunk) is compacted first when the
// floor has risen since its entries were taken (`floor_seen`); otherwise the saturating append runs.
__device__ __forceinline__ void sk_filter_chunk(SkQueue& q, const uint32_t (&r)[kChunk], int nv, int col_chunk,
                                                SkFloor& floor, float& floor_seen, unsigned int* stat,
                                                SkProf* prof = nullptr) {
  bool roomy = __reduce_max_sync(0xffffffffu, q.count()) <= kSkQueue - kChunk;
  if (!roomy && __any_sync(0xffffffffu, floor.keep > floor_seen)) {
    sk_compact(q, floor.keep);
    floor_seen = floor.keep;
    roomy = __reduce_max_sync(0xffffffffu, q.count()) <= kSkQueue - kChunk;
  }
  if (roomy) {
    if (nv >= kChunk) sk_append_roomy<true>(q, r, nv, col_chunk, floor.in);
    else sk_append_roomy<false>(q, r, nv, col_chunk, floor.in);
    return;
  }
  // half a chunk at a time needs only 16 free slots: keeps rows with few lists (20..40 live entries) on the fast form
  const uint32_t wr0 = q.wr;
  if (__reduce_max_sync(0xffffffffu, q.count()) <= kSkQueue - kChunk / 2) {
    sk_append_roomy<false, 0, kChunk / 2>(q, r, nv, col_chunk, floor.in);
    if (__reduce_max_sync(0xffffffffu, q.count()) <= kSkQueue - kChunk / 2) {
      sk_append_roomy<false, kChunk / 2, kChunk>(q, r, nv, col_chunk, floor.in);
      return;
    }
    q.wr = wr0;   // the second half may not fit: take the whole chunk through the saturating form
  }
  if (prof) prof->crowded += 1;
  if (sk_append_sat(q, r, nv, col_chunk, floor.in)) return;
  q.wr = wr0;                                   // a lane ran out of slots: rewind, make room, redo the chunk
  sk_compact(q, floor.keep);
  if (__any_sync(0xffffffffu, q.count() > kSkQueue - kChunk)) sk_select(q, floor, kSkSelectTo, stat, prof);
  floor_seen = floor.keep;
  sk_append_roomy<false>(q, r, nv, col_chunk, floor.in);
}

}  // namespace umma
}  // namespace hgr
