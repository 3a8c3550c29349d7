// Static work decomposition of the fused logit + top-k head (shared by host and device).
//
// The class dimension is cut into UNITS of 16 bank rows (the N granularity of a
// tcgen05.mma with M = 128 / 256).  The (row-tile, unit) space is flattened row-tile-major and
// split into G contiguous, equally sized chunks, one per persistent worker -- a stream-K-style
// split along N.  A worker is one CTA (row tile = 128 image rows) or one CTA PAIR sharing a
// cta_group::2 MMA (row tile = 256 rows).  No fix-up reduction is needed because top-k lists
// merge associatively: every (row-tile, worker) intersection ("segment") emits partial top-K
// lists per row and a small merge kernel combines the lists of a row.
#pragma once
#include <cstdint>

#ifndef __CUDACC__   // host-only unit test of the schedule (g++): the CUDA qualifiers are no-ops
#ifndef __host__
#define __host__
#endif
#ifndef __device__
#define __device__
#endif
#endif

namespace hgr {

constexpr int kTileM = 128;   // image rows per CTA = TMEM lanes
constexpr int kUnit = 16;     // bank rows per scheduling unit
constexpr int kSubN = 256;    // max bank rows per MMA sub-tile (one TMEM accumulator buffer)

struct Sched {
  int32_t G;     // persistent workers (CTAs or CTA pairs)
  int32_t MT;    // row tiles = ceil(B / rows)
  int32_t U;     // units per row tile = ceil(C / 16)
  int32_t P;     // max workers intersecting one row tile
  int32_t rows;  // image rows per row tile: 128 (single CTA) or 256 (CTA pair)
  int64_t T;     // MT * U

  __host__ __device__ int64_t unit_begin(int32_t w) const { return (static_cast<int64_t>(w) * T) / G; }
  // worker whose chunk contains flattened unit x (chunks are non-empty because G <= T)
  __host__ __device__ int32_t owner(int64_t x) const {
    return static_cast<int32_t>(((x + 1) * G - 1) / T);
  }
  __host__ __device__ int32_t first_cta(int32_t mt) const { return owner(static_cast<int64_t>(mt) * U); }
  __host__ __device__ int32_t last_cta(int32_t mt) const { return owner(static_cast<int64_t>(mt + 1) * U - 1); }
  __host__ __device__ int32_t parts(int32_t mt) const { return last_cta(mt) - first_cta(mt) + 1; }
};

inline Sched make_sched(int64_t B, int64_t C, int num_workers, int tile_rows = kTileM) {
  Sched s;
  s.rows = tile_rows;
  s.MT = static_cast<int32_t>((B + tile_rows - 1) / tile_rows);
  s.U = static_cast<int32_t>((C + kUnit - 1) / kUnit);
  s.T = static_cast<int64_t>(s.MT) * s.U;
  s.G = static_cast<int32_t>(s.T < num_workers ? s.T : num_workers);
  if (s.G < 1) s.G = 1;
  s.P = 1;
  for (int32_t mt = 0; mt < s.MT; ++mt) {
    const int32_t p = s.parts(mt);
    if (p > s.P) s.P = p;
  }
  return s;
}

struct SubTile {
  int mt;      // row tile
  int col0;    // first bank row
  int n;       // MMA N (multiple of 16)
  int nvalid;  // bank rows < C inside the sub-tile
  bool first;  // first sub-tile of a (row tile, CTA) segment
  bool last;   // last sub-tile of the segment
  int seq;     // index of the sub-tile inside its segment
  int group;   // group of the sub-tile's bank rows (GroupWalker only)
};

struct TileWalker {
  int64_t u, u_end;
  int U;
  int64_t C;
  bool first;
  int seq;
  __host__ __device__ TileWalker(const Sched& s, int cta, int64_t C_)
      : u(s.unit_begin(cta)), u_end(s.unit_begin(cta + 1)), U(s.U), C(C_), first(true), seq(0) {}
  // Sub-tiles of a segment in ascending column order: full 256-column sub-tiles first, the REMAINDER (segment length
  // mod 256 columns) last -- its short epilogue is then the exposed tail of the worker.
  __host__ __device__ bool next(SubTile& t) {
    if (u >= u_end) return false;
    const int mt = static_cast<int>(u / U);
    int uu = static_cast<int>(u - static_cast<int64_t>(mt) * U);
    constexpr int kFull = kSubN / kUnit;
    int64_t seg = U - uu;                          // units left in this segment
    if (u_end - u < seg) seg = u_end - u;
    const int nu = seg < kFull ? static_cast<int>(seg) : kFull;
    seq = first ? 0 : seq + 1;
    t.seq = seq;
    t.mt = mt;
    t.col0 = uu * kUnit;
    t.n = nu * kUnit;
    const int64_t left = C - t.col0;
    t.nvalid = left < t.n ? static_cast<int>(left) : t.n;
    t.first = first;
    u += nu;
    uu += nu;
    t.last = (u >= u_end) || (uu == U);
    first = t.last;
    return true;
  }
};

// ---- grouped schedule (hgr_score_topk_splits) ----------------------------------------------------------------------
// The bank rows are cut into n <= 16 contiguous GROUPS [end[g-1], end[g]) (rows of equal split membership), and no
// partial list may hold rows of two groups: then the lists of a row that cover one split are exactly those of its
// groups.  Units are counted per group -- group g has ceil(C_g / 16) units, the first starting at the group's first
// bank row, so a unit may begin at any row -- and the flattened space is (row tile, group, unit): U = sum of the
// groups' units.  The chunks of the workers are cut from that space exactly as in the plain schedule; a segment also
// ends where a group ends.  The table sits next to the Sched instead of inside it, so the parameter block and the code
// of the ungrouped kernels stay as they are.  With n == 1 everything below reduces to the plain schedule.
constexpr int kMaxGroups = 16;

struct Groups {
  int32_t n;                      // groups (1: the plain schedule)
  int32_t end[kMaxGroups];        // exclusive last bank row of group g: strictly ascending, end[n - 1] = C
  int32_t ubeg[kMaxGroups + 1];   // first tile-local unit of group g; ubeg[n] = U

  __host__ __device__ int32_t begin(int g) const { return g > 0 ? end[g - 1] : 0; }
};

// Fills g->ubeg; false when the table is malformed (n outside [1, 16], empty group, end[n - 1] != C).
inline bool make_groups(int64_t C, int n, const int32_t* end, Groups* g) {
  if (n < 1 || n > kMaxGroups) return false;
  g->n = n;
  int64_t prev = 0, units = 0;
  for (int i = 0; i < n; ++i) {
    if (end[i] <= prev) return false;
    g->end[i] = end[i];
    g->ubeg[i] = static_cast<int32_t>(units);
    units += (end[i] - prev + kUnit - 1) / kUnit;
    prev = end[i];
  }
  for (int i = n; i <= kMaxGroups; ++i) g->ubeg[i] = static_cast<int32_t>(units);   // (every word set: tables compare)
  for (int i = n; i < kMaxGroups; ++i) g->end[i] = static_cast<int32_t>(C);
  return prev == C;
}

// List slots of row tile mt are dense and in column order: a new slot starts at every chunk boundary and at every
// group start inside the tile, counted once where the two coincide.  Slot of the segment holding flattened unit x of
// group g (x inside row tile mt):
__host__ __device__ inline int group_slot(const Sched& s, const Groups& gr, int32_t mt, int64_t x, int g) {
  const int64_t t0 = static_cast<int64_t>(mt) * s.U;
  int slot = s.owner(x) - s.first_cta(mt) + g;
  for (int h = 1; h <= g; ++h) {
    const int64_t xh = t0 + gr.ubeg[h];
    if (s.owner(xh - 1) != s.owner(xh)) --slot;   // this group start is also a chunk start
  }
  return slot;
}
__host__ __device__ inline int group_first_slot(const Sched& s, const Groups& gr, int32_t mt, int g) {
  return group_slot(s, gr, mt, static_cast<int64_t>(mt) * s.U + gr.ubeg[g], g);
}
__host__ __device__ inline int group_parts(const Sched& s, const Groups& gr, int32_t mt) {
  return group_slot(s, gr, mt, static_cast<int64_t>(mt + 1) * s.U - 1, gr.n - 1) + 1;
}
// Bank rows [c0, c1) of slot p of row tile mt, given its group g and that group's first slot.
__host__ __device__ inline void group_slot_cols(const Sched& s, const Groups& gr, int32_t mt, int p, int g, int first,
                                                int64_t& c0, int64_t& c1) {
  const int64_t t0 = static_cast<int64_t>(mt) * s.U;
  const int w = s.owner(t0 + gr.ubeg[g]) + (p - first);   // every later slot of the group starts a new chunk
  int64_t u0 = p == first ? gr.ubeg[g] : s.unit_begin(w) - t0;
  int64_t u1 = s.unit_begin(w + 1) - t0;
  u1 = u1 < gr.ubeg[g + 1] ? u1 : gr.ubeg[g + 1];
  c0 = gr.begin(g) + (u0 - gr.ubeg[g]) * kUnit;
  c1 = gr.begin(g) + (u1 - gr.ubeg[g]) * kUnit;
  c1 = c1 < gr.end[g] ? c1 : gr.end[g];
}
// Group and bank rows of slot p of row tile mt (p < group_parts).
__host__ __device__ inline int group_slot_range(const Sched& s, const Groups& gr, int32_t mt, int p, int64_t& c0,
                                                int64_t& c1) {
  int g = 0, first = 0;
  for (int h = 1; h < gr.n; ++h) {
    const int f = group_first_slot(s, gr, mt, h);
    if (f > p) break;
    g = h;
    first = f;
  }
  group_slot_cols(s, gr, mt, p, g, first, c0, c1);
  return g;
}

// Sched over the units of a group table: G, MT, U, T as make_sched over U units, P = the most slots of a row tile.
inline Sched make_sched_groups(int64_t B, const Groups& gr, int num_workers, int tile_rows) {
  Sched s = make_sched(B, static_cast<int64_t>(gr.ubeg[gr.n]) * kUnit, num_workers, tile_rows);
  s.P = 1;
  for (int32_t mt = 0; mt < s.MT; ++mt) {
    const int p = group_parts(s, gr, mt);
    if (p > s.P) s.P = p;
  }
  return s;
}

// TileWalker over the grouped schedule: a segment also ends at the end of a group, `nvalid` masks the columns past
// the group's end (rows of the next group, loaded but never emitted), t.group names the group.
struct GroupWalker {
  int64_t u, u_end;
  int U;
  const Groups* gr;
  int g;
  bool first;
  int seq;
  __host__ __device__ GroupWalker(const Sched& s, int cta, const Groups& groups)
      : u(s.unit_begin(cta)), u_end(s.unit_begin(cta + 1)), U(s.U), gr(&groups), g(0), first(true), seq(0) {}
  __host__ __device__ bool next(SubTile& t) {
    if (u >= u_end) return false;
    const int mt = static_cast<int>(u / U);
    int uu = static_cast<int>(u - static_cast<int64_t>(mt) * U);
    if (first) {
      g = 0;
      while (uu >= gr->ubeg[g + 1]) ++g;
    }
    constexpr int kFull = kSubN / kUnit;
    int64_t seg = gr->ubeg[g + 1] - uu;            // units left in this segment
    if (u_end - u < seg) seg = u_end - u;
    const int nu = seg < kFull ? static_cast<int>(seg) : kFull;
    seq = first ? 0 : seq + 1;
    t.seq = seq;
    t.mt = mt;
    t.group = g;
    t.col0 = gr->begin(g) + (uu - gr->ubeg[g]) * kUnit;
    t.n = nu * kUnit;
    const int left = gr->end[g] - t.col0;
    t.nvalid = left < t.n ? left : t.n;
    t.first = first;
    u += nu;
    uu += nu;
    t.last = (u >= u_end) || (uu == gr->ubeg[g + 1]);
    first = t.last;
    return true;
  }
  // flattened unit of a sub-tile's first column (for group_slot)
  __host__ __device__ int64_t unit_of(const SubTile& t) const {
    return static_cast<int64_t>(t.mt) * U + gr->ubeg[t.group] + (t.col0 - gr->begin(t.group)) / kUnit;
  }
};

}  // namespace hgr
