// Host-side exhaustive check of the static schedule (hgrnet_b200/csrc/sched.cuh), compiled with g++ by
// tests/test_cpu_sched.py.  For every (B, C, workers, rows-per-tile) on the command line it walks every worker's
// chunk with the SAME TileWalker the kernels use and verifies:
//   * every (row tile, bank row) is covered exactly once, by sub-tiles of <= 256 rows in units of 16;
//   * nvalid clips the last unit at C; first / last / seq flags delimit segments; a segment never crosses a row tile;
//   * the partial-list slot of a segment (worker - first_cta(row tile)) is unique inside [0, parts(row tile));
//   * owner() inverts unit_begin(), chunks are non-empty and ordered, P = max parts.
// Prints "ok <n_checked>" or a message and exits non-zero.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../hgrnet_b200/csrc/sched.cuh"

using namespace hgr;

static int fail(const char* what, long long B, long long C, int G, int rows) {
  std::printf("FAIL %s at B=%lld C=%lld workers=%d rows=%d\n", what, B, C, G, rows);
  return 1;
}

static int check(long long B, long long C, int workers, int rows) {
  const Sched s = make_sched(B, C, workers, rows);
  if (s.G < 1 || s.G > workers || s.G > s.T) return fail("G range", B, C, workers, rows);
  if (s.unit_begin(0) != 0 || s.unit_begin(s.G) != s.T) return fail("chunk ends", B, C, workers, rows);
  int maxp = 0;
  for (int mt = 0; mt < s.MT; ++mt) {
    if (s.parts(mt) < 1) return fail("parts < 1", B, C, workers, rows);
    maxp = s.parts(mt) > maxp ? s.parts(mt) : maxp;
  }
  if (maxp != s.P) return fail("P != max parts", B, C, workers, rows);
  std::vector<unsigned char> cover(static_cast<size_t>(s.MT) * s.U, 0);
  std::vector<unsigned char> slot_used(static_cast<size_t>(s.MT) * s.P, 0);
  for (int w = 0; w < s.G; ++w) {
    const long long b = s.unit_begin(w), e = s.unit_begin(w + 1);
    if (e <= b) return fail("empty chunk", B, C, workers, rows);
    if (s.owner(b) != w || s.owner(e - 1) != w) return fail("owner != worker", B, C, workers, rows);
    TileWalker walk(s, w, C);
    SubTile t;
    bool open = false;
    int seq = 0, seg_mt = -1;
    long long next_unit = b;
    while (walk.next(t)) {
      if (t.n <= 0 || t.n > kSubN || t.n % kUnit) return fail("sub-tile size", B, C, workers, rows);
      if (t.col0 % kUnit) return fail("col0 alignment", B, C, workers, rows);
      if (t.mt < 0 || t.mt >= s.MT) return fail("row tile range", B, C, workers, rows);
      const long long u0 = static_cast<long long>(t.mt) * s.U + t.col0 / kUnit;
      if (u0 != next_unit) return fail("sub-tiles not contiguous", B, C, workers, rows);
      next_unit += t.n / kUnit;
      if (t.col0 / kUnit + t.n / kUnit > s.U) return fail("sub-tile crosses a row tile", B, C, workers, rows);
      const long long left = C - t.col0;
      const int nv = left < t.n ? static_cast<int>(left) : t.n;
      if (t.nvalid != nv || nv <= 0) return fail("nvalid", B, C, workers, rows);
      if (t.first != !open) return fail("first flag", B, C, workers, rows);
      if (t.first) {
        seq = 0;
        seg_mt = t.mt;
        const int slot = w - s.first_cta(t.mt);
        if (slot < 0 || slot >= s.parts(t.mt)) return fail("slot range", B, C, workers, rows);
        unsigned char& used = slot_used[static_cast<size_t>(t.mt) * s.P + slot];
        if (used) return fail("slot used twice", B, C, workers, rows);
        used = 1;
      }
      if (t.mt != seg_mt) return fail("segment crosses a row tile", B, C, workers, rows);
      if (t.seq != seq++) return fail("seq", B, C, workers, rows);
      for (int k = 0; k < t.n / kUnit; ++k) {
        unsigned char& c = cover[static_cast<size_t>(u0) + k];
        if (c) return fail("unit covered twice", B, C, workers, rows);
        c = 1;
      }
      open = !t.last;
    }
    if (open) return fail("segment left open", B, C, workers, rows);
    if (next_unit != e) return fail("chunk not exhausted", B, C, workers, rows);
  }
  for (size_t i = 0; i < cover.size(); ++i)
    if (!cover[i]) return fail("unit not covered", B, C, workers, rows);
  for (int mt = 0; mt < s.MT; ++mt)
    for (int p = 0; p < s.parts(mt); ++p)
      if (!slot_used[static_cast<size_t>(mt) * s.P + p]) return fail("slot never written", B, C, workers, rows);
  return 0;
}

int main(int argc, char** argv) {
  long long n = 0;
  for (int i = 1; i + 3 < argc; i += 4) {
    const long long B = std::atoll(argv[i]), C = std::atoll(argv[i + 1]);
    const int workers = std::atoi(argv[i + 2]), rows = std::atoi(argv[i + 3]);
    if (check(B, C, workers, rows)) return 1;
    ++n;
  }
  std::printf("ok %lld\n", n);
  return 0;
}
