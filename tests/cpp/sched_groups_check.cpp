// Host-side exhaustive check of the GROUPED schedule (hgrnet_b200/csrc/sched.cuh: Groups, GroupWalker, group_slot*),
// compiled with g++ by tests/test_cpu_sched_groups.py.  Arguments: cases of the form
//   B workers rows n end[0] ... end[n-1]        (C = end[n-1])
// For every case it walks every worker's chunk with the SAME GroupWalker the kernels use and verifies:
//   * every (row tile, bank row < C) pair is covered exactly once, by sub-tiles of <= 256 rows in units of 16;
//   * no segment crosses the end of a group, nvalid clips every sub-tile at its group's end;
//   * the list slots of a row tile are dense, unique and in column order (group_slot, group_parts, P = max);
//   * group_slot_range recovers for every slot the group and the bank rows the walker emitted into it;
//   * with one group: make_sched_groups == make_sched and the walk is the TileWalker's, sub-tile by sub-tile.
// Prints "ok <n_checked>" or a message and exits non-zero.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../hgrnet_b200/csrc/sched.cuh"

using namespace hgr;

static int fail(const char* what, long long B, long long C, int G, int rows, int n) {
  std::printf("FAIL %s at B=%lld C=%lld workers=%d rows=%d groups=%d\n", what, B, C, G, rows, n);
  return 1;
}

struct Seg {
  long long c0 = -1, c1 = -1;
  int g = -1;
  bool used = false;
};

static int check(long long B, int workers, int rows, int n, const int32_t* end) {
  const long long C = end[n - 1];
#define FAIL(what) return fail(what, B, C, workers, rows, n)
  Groups gr;
  if (!make_groups(C, n, end, &gr)) FAIL("make_groups rejected a valid table");
  const Sched s = make_sched_groups(B, gr, workers, rows);
  if (s.G < 1 || s.G > workers || s.G > s.T) FAIL("G range");
  if (s.unit_begin(0) != 0 || s.unit_begin(s.G) != s.T) FAIL("chunk ends");
  if (n == 1) {
    const Sched p = make_sched(B, C, workers, rows);
    if (p.G != s.G || p.MT != s.MT || p.U != s.U || p.P != s.P || p.rows != s.rows || p.T != s.T)
      FAIL("one group: schedule differs from make_sched");
    for (int mt = 0; mt < s.MT; ++mt)
      if (group_parts(s, gr, mt) != p.parts(mt)) FAIL("one group: slots differ from parts()");
  }
  int maxp = 0;
  for (int mt = 0; mt < s.MT; ++mt) maxp = group_parts(s, gr, mt) > maxp ? group_parts(s, gr, mt) : maxp;
  if (maxp != s.P) FAIL("P != max slots");
  std::vector<unsigned char> cover(static_cast<size_t>(s.MT) * C, 0);
  std::vector<Seg> segs(static_cast<size_t>(s.MT) * s.P);
  for (int w = 0; w < s.G; ++w) {
    GroupWalker walk(s, w, gr);
    TileWalker plain(s, w, C);
    SubTile t, pt;
    bool open = false;
    int seq = 0, seg_mt = -1, seg_g = -1;
    Seg* cur = nullptr;
    long long next_col = -1;
    while (walk.next(t)) {
      if (n == 1) {
        if (!plain.next(pt)) FAIL("one group: walk longer than the TileWalker's");
        if (pt.mt != t.mt || pt.col0 != t.col0 || pt.n != t.n || pt.nvalid != t.nvalid || pt.first != t.first ||
            pt.last != t.last || pt.seq != t.seq)
          FAIL("one group: sub-tile differs from the TileWalker's");
      }
      if (t.n <= 0 || t.n > kSubN || t.n % kUnit) FAIL("sub-tile size");
      if (t.mt < 0 || t.mt >= s.MT) FAIL("row tile range");
      if (t.group < 0 || t.group >= n) FAIL("group range");
      if (t.col0 < gr.begin(t.group) || t.col0 >= gr.end[t.group]) FAIL("sub-tile starts outside its group");
      if ((t.col0 - gr.begin(t.group)) % kUnit) FAIL("col0 not on a unit of its group");
      const long long nv = std::min<long long>(t.n, gr.end[t.group] - t.col0);
      if (t.nvalid != nv || nv <= 0) FAIL("nvalid");
      if (t.first != !open) FAIL("first flag");
      if (t.first) {
        seq = 0;
        seg_mt = t.mt;
        seg_g = t.group;
        const int slot = group_slot(s, gr, t.mt, walk.unit_of(t), t.group);
        if (slot < 0 || slot >= group_parts(s, gr, t.mt)) FAIL("slot range");
        cur = &segs[static_cast<size_t>(t.mt) * s.P + slot];
        if (cur->used) FAIL("slot used twice");
        cur->used = true;
        cur->c0 = t.col0;
        cur->g = t.group;
        next_col = t.col0;
      } else {
        if (t.col0 != next_col) FAIL("sub-tiles of a segment not contiguous");
      }
      if (t.mt != seg_mt) FAIL("segment crosses a row tile");
      if (t.group != seg_g) FAIL("segment crosses a group end");
      if (t.seq != seq++) FAIL("seq");
      for (int k = 0; k < t.nvalid; ++k) {
        unsigned char& c = cover[static_cast<size_t>(t.mt) * C + t.col0 + k];
        if (c) FAIL("bank row covered twice");
        c = 1;
      }
      next_col = t.col0 + t.n;
      cur->c1 = t.col0 + t.nvalid;
      open = !t.last;
    }
    if (n == 1 && plain.next(pt)) FAIL("one group: walk shorter than the TileWalker's");
    if (open) FAIL("segment left open");
  }
  for (size_t i = 0; i < cover.size(); ++i)
    if (!cover[i]) FAIL("bank row not covered");
  for (int mt = 0; mt < s.MT; ++mt) {
    long long prev_end = 0;
    for (int p = 0; p < group_parts(s, gr, mt); ++p) {
      const Seg& sg = segs[static_cast<size_t>(mt) * s.P + p];
      if (!sg.used) FAIL("slot never written");
      if (sg.c0 != prev_end) FAIL("slots not in column order");
      prev_end = sg.c1;
      int64_t c0 = 0, c1 = 0;
      const int g = group_slot_range(s, gr, mt, p, c0, c1);
      if (g != sg.g || c0 != sg.c0 || c1 != sg.c1) FAIL("group_slot_range differs from the walk");
    }
    if (prev_end != C) FAIL("slots do not end at C");
  }
  return 0;
#undef FAIL
}

int main(int argc, char** argv) {
  long long cases = 0;
  int i = 1;
  while (i + 3 < argc) {
    const long long B = std::atoll(argv[i]);
    const int workers = std::atoi(argv[i + 1]), rows = std::atoi(argv[i + 2]), n = std::atoi(argv[i + 3]);
    i += 4;
    if (n < 1 || n > kMaxGroups || i + n > argc) {
      std::printf("FAIL bad case %lld\n", cases);
      return 1;
    }
    std::vector<int32_t> end(n);
    for (int g = 0; g < n; ++g) end[g] = std::atoi(argv[i + g]);
    i += n;
    if (check(B, workers, rows, n, end.data())) return 1;
    ++cases;
  }
  std::printf("ok %lld\n", cases);
  return 0;
}
