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

}  // namespace hgr
