"""Ordered banks reach the overflow branches of the deferred-insert top-K epilogue (``score_pair.cu``:
``epi_topk_defer``), checked without a GPU.

The bit-for-bit grid of ``tests/test_gpu_topk_exact.py`` runs on banks in random row order, where a row's survivors
rarely fill the candidate queue.  Real banks are in tree order: a row's best classes come in runs.  This file builds
ordered banks on the host (``(X, bank)`` in bf16 from a CPU generator, the exact inputs ``tests/test_gpu_topk_ordered.py``
hands the kernels) and restates, in float64, the walk of one worker (``sched.cuh``) and the queue accounting of the
epilogue (warm-up floor, the sub-tile threshold, the per-chunk branch, the drain at the end of a sub-tile) for sampled
warps.  A comparison counts only when it is decided by the error bound of ``check_topk_f64`` (an fp32 sum of D
products is within ``(D + 2) 2^-23 |x|.|w|`` of the float64 logit); a warp with an undecided comparison is not used as
evidence.  The queue lengths, the chunk and sub-tile widths and the early-drain rule are read from the CUDA sources,
so a kernel change moves the model with it.  The sets asserted below are the branches the GPU test claims to cover."""
from __future__ import annotations

import os
import re

import numpy as np
import pytest
import torch

from tests.util import _unit_bf16, hostile_bank

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hgrnet_b200", "csrc")
PAIRS = 74                                # CTA pairs of 148 SMs (the sketch and the grouped schedule use all)


def _ops():
    """The host-side plan (``ops.score_topk_plan`` / ``ops.global_list_len``; 148 SMs when no device is visible)."""
    from hgrnet_b200 import ops
    return ops


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _int(pattern, text):
    m = re.search(pattern, text)
    assert m, pattern
    return [int(g) for g in m.groups()]


def kernel_consts():
    """Widths and queue rules of the kernel, read from its sources."""
    um, sc, sp = _src("umma_common.cuh"), _src("sched.cuh"), _src("score_pair.cu")
    narrow, q_narrow, q_wide = _int(r"defer_queue_len\(\)\s*\{\s*return\s+KL\s*<=\s*(\d+)\s*\?\s*(\d+)\s*:\s*(\d+)\s*;",
                                    um)
    (drain_above,) = _int(r"if\s*\(\s*!roomy\s*&&\s*KL\s*>\s*(\d+)\s*\)", sp)
    (chunk,) = _int(r"constexpr int kChunk\s*=\s*(\d+);", um)
    (unit,) = _int(r"constexpr int kUnit\s*=\s*(\d+);", sc)
    (sub_n,) = _int(r"constexpr int kSubN\s*=\s*(\d+);", sc)
    return dict(narrow=narrow, q_narrow=q_narrow, q_wide=q_wide, drain_above=drain_above, chunk=chunk, unit=unit,
                sub_n=sub_n)


KC = kernel_consts()
UNIT, SUB_N, CHUNK = KC["unit"], KC["sub_n"], KC["chunk"]
RUN = 2 * SUB_N               # a rising run: two full sub-tiles
DIP = SUB_N + 6 * CHUNK       # the last two chunks of a run lie below all the rest of it


def queue_len(KL):
    return KC["q_narrow"] if KL <= KC["narrow"] else KC["q_wide"]


def exact_len(K):
    return 8 if K <= 8 else 12 if K <= 12 else 20 if K <= 20 else 32


# ---- schedule (sched.cuh) -------------------------------------------------------------------------------------------

def make_sched(B, C, workers, rows=256, units=None):
    MT, U = -(-B // rows), (-(-C // UNIT) if units is None else units)
    T = MT * U
    return dict(G=max(1, min(T, workers)), MT=MT, U=U, T=T, rows=rows)


def owner(s, x):
    return ((x + 1) * s["G"] - 1) // s["T"]


def first_cta(s, mt):
    return owner(s, mt * s["U"])


def parts(s, mt):
    return owner(s, (mt + 1) * s["U"] - 1) - first_cta(s, mt) + 1


def walk(s, C, w):
    """Sub-tiles of worker w (TileWalker::next): dict(mt, col0, n, nvalid, first, last, seq)."""
    G, U, T = s["G"], s["U"], s["T"]
    u, u_end, first, seq = w * T // G, (w + 1) * T // G, True, 0
    while u < u_end:
        mt, uu = divmod(u, U)
        nu = min(U - uu, u_end - u, SUB_N // UNIT)
        seq = 0 if first else seq + 1
        col0, n = uu * UNIT, nu * UNIT
        u, uu = u + nu, uu + nu
        last = u >= u_end or uu == U
        yield dict(mt=mt, col0=col0, n=n, nvalid=min(n, C - col0), first=first, last=last, seq=seq, group=0)
        first = last


def group_units(ends):
    ubeg, prev = [0], 0
    for e in ends:
        ubeg.append(ubeg[-1] + -(-(e - prev) // UNIT))
        prev = e
    return ubeg


def walk_groups(s, ends, w):
    """Sub-tiles of worker w on the grouped schedule (GroupWalker::next)."""
    ubeg = group_units(ends)
    begin = [0] + list(ends[:-1])
    G, U, T = s["G"], s["U"], s["T"]
    u, u_end, first, seq, g = w * T // G, (w + 1) * T // G, True, 0, 0
    while u < u_end:
        mt, uu = divmod(u, U)
        if first:
            g = 0
            while uu >= ubeg[g + 1]:
                g += 1
        nu = min(ubeg[g + 1] - uu, u_end - u, SUB_N // UNIT)
        seq = 0 if first else seq + 1
        col0, n = begin[g] + (uu - ubeg[g]) * UNIT, nu * UNIT
        u, uu = u + nu, uu + nu
        last = u >= u_end or uu == ubeg[g + 1]
        yield dict(mt=mt, col0=col0, n=n, nvalid=min(n, ends[g] - col0), first=first, last=last, seq=seq, group=g)
        first = last


def segments(tiles):
    """Split a worker's sub-tiles into its segments (a segment ends at a `last` sub-tile)."""
    seg = []
    for t in tiles:
        seg.append(t)
        if t["last"]:
            yield seg
            seg = []


def plan_sched(B, C, D, K):
    return make_sched(B, C, _ops().score_topk_plan(B, C, D, K)["workers"])


def row_tile_segments(s, C, mt, walker=None):
    """(worker, first column, end column) of every segment of row tile mt."""
    out = []
    for w in range(first_cta(s, mt), first_cta(s, mt) + parts(s, mt)):
        for seg in segments(walker(w) if walker else walk(s, C, w)):
            if seg[0]["mt"] == mt:
                out.append((w, seg[0]["col0"], seg[-1]["col0"] + seg[-1]["nvalid"]))
    return out


# ---- ordered banks, seeded on the host ------------------------------------------------------------------------------

# (B, C, D, K) of every case.  Production / exact list lengths (148 SMs):
SHAPES = {
    "cfg2": (512, 21841, 1024, 20),     # production 8, exact 20
    "cfg2_k8": (512, 21841, 1024, 8),   # exact 8
    "kl10": (257, 21841, 256, 21),      # production 10, exact 32
    "k12": (1024, 10921, 256, 12),      # production 8, exact 12
    "kl12": (1024, 10921, 256, 21),     # production 12, exact 32
    "kl16": (1024, 10921, 256, 32),     # production 16, exact 32
    "kl32": (2047, 5461, 256, 32),      # production = exact 32
    "cfg5": (4096, 21841, 1024, 20),    # production = exact 20 (B = 4096)
    "shard": (4096, 2731, 1024, 20),    # one class shard of eight: global list length 10 for C_total = 8 C
}
SHARD_N = 8
# kinds per shape: every shape has rising runs; the speculative shapes also the certified kind
KINDS = {
    "cfg2": ("rising", "rising_below_top", "tied", "tree"),
    "cfg2_k8": ("rising",),
    "kl10": ("rising", "rising_below_top", "tree"),
    "k12": ("rising", "rising_below_top"),
    "kl12": ("rising", "rising_below_top"),
    "kl16": ("rising", "rising_below_top", "tied"),
    "kl32": ("rising", "tied"),
    "cfg5": ("rising", "tied", "tree"),
    "shard": ("rising",),
}
# grouped schedule: three groups (split 0 = groups 0 and 1, split 1 = groups 1 and 2); one rising run crosses the end of
# group 0, one fills group 2
SPLIT_SHAPE = (4096, 2731, 256)
SPLIT_ENDS = [1000, 2200, 2731]
SPLIT_MASKS = [0b01, 0b11, 0b10]
SPLIT_RUNS = [(600, 1400), (2200, 2731)]
SPLIT_KS = (8, 20)


def _orth(g, u, n):
    v = torch.randn(n, u.numel(), generator=g, dtype=torch.float64)
    v = v - (v @ u)[:, None] * u[None, :]
    return v / v.norm(dim=1, keepdim=True)


def _aligned(g, u, c):
    """Unit rows at cosine c[i] from u in the plane of u and one direction v orthogonal to u: a query x near u sees
    c (x.u) + sqrt(1 - c^2) (x.v), monotone in c while x.v is small."""
    c = torch.as_tensor(c, dtype=torch.float64)
    v = _orth(g, u, 1)
    return c[:, None] * u[None, :] + (1 - c * c).clamp_min(0).sqrt()[:, None] * v


def run_segments(s, C, need=RUN):
    """Segments of row tile 0 long enough for a run (two full sub-tiles and a later one): the first and a middle one."""
    segs = [(a, e) for _, a, e in row_tile_segments(s, C, 0) if e - a >= need]
    assert segs, "no segment of row tile 0 holds a run"
    return sorted({segs[0], segs[len(segs) // 2]})


def build(kind, B, C, D, K, sched, runs=None, seed=0):
    """``(X, bank, info)``: bf16 CPU tensors and where the runs / top rows / tied copies are.

    rising -- along each run the rows are ``normalize(c u + s v + noise)`` with c rising from 0.35 to 0.93, every query
    is near u, so every row's logits rise by about 1e-3 per column, far above the fp32 error bound; the rest is random.
    The last two chunks of the second sub-tile dip below the whole run (c from 0.30 to 0.34): the queue then holds
    the redone chunk before them and takes the saturating append that fits.  The run's largest values come in the sixth
    chunk of that sub-tile, a failed and redone append; a kernel that lost the redo would drop every odd chunk there
    (the queue is empty after each failed append, so the next chunk is roomy), and with it every row's best values.
    rising_below_top -- the same, plus K top rows (c in [0.985, 0.999]) that beat every run value, spread evenly over
    the columns outside the runs' segments.  tied -- K - 1 top rows; the first run segment rises over its first
    sub-tile (c from 0.35 to 0.6) and its second sub-tile holds copies of one row (c = 0.96): their value is every
    row's K-th, the tie is cut at the first copy.  tree --
    ``hostile_bank("clustered")`` (siblings adjacent and similar) with queries near random bank rows."""
    g = torch.Generator().manual_seed(1000 * seed + B + C + D + K)
    if kind == "tree":
        bank = hostile_bank(C, D, "clustered", seed=5)
        pick = torch.randint(0, C, (B,), generator=g)
        X = _unit_bf16(bank[pick].double() + 0.3 * torch.randn(B, D, generator=g, dtype=torch.float64) / D ** 0.5)
        return X, bank, dict(runs=[], top=[], tied=[])
    u = torch.randn(D, generator=g, dtype=torch.float64)
    u = u / u.norm()
    w = torch.randn(C, D, generator=g, dtype=torch.float64)
    if runs is None:
        runs = [(a, min(a + RUN, e)) for a, e in run_segments(sched, C)]
    info = dict(runs=[], top=[], tied=[])
    if kind in ("rising", "rising_below_top"):
        for a, e in runs:
            c = torch.linspace(0.35, 0.93, e - a, dtype=torch.float64)
            if e - a >= DIP + 2 * CHUNK:
                c[DIP:DIP + 2 * CHUNK] = torch.linspace(0.30, 0.34, 2 * CHUNK, dtype=torch.float64)
            w[a:e] = _aligned(g, u, c) + 0.003 * torch.randn(e - a, D, generator=g, dtype=torch.float64) / D ** 0.5
            info["runs"].append((a, e))
    if kind in ("rising_below_top", "tied"):
        n_top = K if kind == "rising_below_top" else K - 1
        busy = set()
        for a, e in run_segments(sched, C):
            busy |= set(range(a - SUB_N, e + SUB_N))
        free = [c for c in range(C) if c not in busy]
        top = [free[(2 * i + 1) * len(free) // (2 * n_top)] for i in range(n_top)]
        cos = 0.985 + 0.014 * torch.rand(n_top, generator=g, dtype=torch.float64)
        w[top] = _aligned(g, u, cos)
        info["top"] = top
    if kind == "tied":
        a, _ = run_segments(sched, C)[0]
        w[a:a + SUB_N] = _aligned(g, u, torch.linspace(0.35, 0.6, SUB_N, dtype=torch.float64))
        copies = list(range(a + SUB_N, a + 2 * SUB_N))
        w[copies] = _aligned(g, u, [0.96])[0]
        info["tied"] = copies
    bank = _unit_bf16(w)
    X = _unit_bf16(u[None, :] + 0.3 * torch.randn(B, D, generator=g, dtype=torch.float64) / D ** 0.5)
    return X, bank, info


def build_splits(K, seed=0):
    B, C, D = SPLIT_SHAPE
    s = splits_sched()
    return build("rising", B, C, D, K, s, runs=SPLIT_RUNS, seed=seed)


def splits_sched():
    B, C, _ = SPLIT_SHAPE
    return make_sched(B, C, PAIRS, units=group_units(SPLIT_ENDS)[-1])


def build_shard(seed=0):
    B, C, D, K = SHAPES["shard"]
    return build("rising", B, C, D, K, plan_sched(B, C, D, K), seed=seed)


def case_inputs(name, kind):
    B, C, D, K = SHAPES[name]
    return build(kind, B, C, D, K, plan_sched(B, C, D, K))


# ---- the queue accounting of epi_topk_defer, in float64 -------------------------------------------------------------

class Undecided(Exception):
    pass


class WarpModel:
    """The 32 rows of one epilogue warp over one worker's segment.  Columns are indices into the segment."""

    def __init__(self, X, W, canon, KL):
        x, w = X.double(), W.double()
        self.R = (x @ w.T).numpy()
        self.E = ((X.shape[1] + 2) * 2.0 ** -23 * (x.abs() @ w.abs().T)).numpy()
        self.lo, self.hi = self.R - self.E, self.R + self.E
        self.canon = canon
        self.KL = KL

    def cmp(self, l, a, b):
        """Sign of value(a) - value(b) in row l for column array a and column b, where decided: equal for copies of
        one bank row (or exact zeros); else the float64 intervals must not overlap."""
        eq = (self.canon[a] == self.canon[b]) | ((self.E[l, a] == 0) & (self.E[l, b] == 0) &
                                                  (self.R[l, a] == self.R[l, b]))
        gt = self.lo[l, a] > self.hi[l, b]
        lt = self.hi[l, a] < self.lo[l, b]
        if not (eq | gt | lt).all():
            raise Undecided
        return np.where(eq, 0, np.where(gt, 1, -1))

    def _by_value(self, l, cols):
        return cols[np.lexsort((cols, -self.R[l, cols]))]

    def warmup_floor(self, l, cols, nvalid):
        """warmup_floor_pairs: the column whose value is tau (x > floor <=> x >= tau), or None (-inf)."""
        if nvalid < CHUNK:
            return None
        full = cols[:nvalid // CHUNK * CHUNK]
        G = self.KL // 2
        grp = (np.arange(full.size) % CHUNK) % G
        second = [self._by_value(l, full[grp == h])[1] for h in range(G)]
        tau = second[int(np.argmin([self.R[l, c] for c in second]))]
        for h in range(G):
            r = self.cmp(l, full[grp == h], tau)
            if (r >= 0).sum() < 2 or (h == grp[np.searchsorted(full, tau)] and (r > 0).sum() > 1):
                raise Undecided
        return tau

    def list_thr(self, l, S):
        """The list's KL-th entry over the drained columns S (a column, or None while not full); prunes S."""
        if S.size < self.KL:
            return None, S
        c = self._by_value(l, S)[self.KL - 1]
        r = self.cmp(l, S, c)
        if not ((r > 0).sum() < self.KL <= (r >= 0).sum()):
            raise Undecided
        return c, S[r >= 0]

    def passes(self, l, cols, floor, thr):
        ok = np.ones(cols.size, bool)
        if floor is not None:
            ok &= self.cmp(l, cols, floor) >= 0
        if thr is not None:
            ok &= self.cmp(l, cols, thr) > 0
        return ok

    def run(self, tiles, base):
        """Branches taken over the sub-tiles of one segment: a set of (later, branch); None when undecided."""
        L, KL = queue_len(self.KL), self.KL
        ev = set()
        try:
            S = [np.zeros(0, np.int64) for _ in range(32)]
            floor = [None] * 32
            for t in tiles:
                cols = np.arange(t["col0"] - base, t["col0"] - base + t["nvalid"])
                later = not t["first"]
                if t["first"]:
                    floor = [self.warmup_floor(l, cols, t["nvalid"]) for l in range(32)]
                thr = [None] * 32
                for l in range(32):
                    thr[l], S[l] = self.list_thr(l, S[l])
                queue = [[] for _ in range(32)]

                def drain():
                    for l in range(32):
                        if queue[l]:
                            S[l] = np.concatenate([S[l]] + queue[l])
                            queue[l] = []
                        thr[l], S[l] = self.list_thr(l, S[l])

                def survivors(ch):
                    return [ch[self.passes(l, ch, floor[l], thr[l])] for l in range(32)]

                for c0 in range(0, t["nvalid"], CHUNK):
                    ch = cols[c0:c0 + CHUNK]
                    count = np.array([sum(q.size for q in queue[l]) for l in range(32)])
                    roomy = count.max() <= L - CHUNK
                    if not roomy and KL > KC["drain_above"]:
                        ev.add((later, "early_drain"))
                        drain()
                    elif roomy or KL > KC["drain_above"]:
                        ev.add((later, "roomy"))
                    else:
                        sv = survivors(ch)
                        if (count + np.array([v.size for v in sv]) >= L).any():
                            ev.add((later, "fail_redo"))
                            drain()
                            sv = survivors(ch)
                            if max(v.size for v in sv) >= L:
                                ev.add((later, "reload"))
                                for l in range(32):
                                    S[l] = np.concatenate([S[l], sv[l]])
                                    thr[l], S[l] = self.list_thr(l, S[l])
                                continue
                        else:
                            ev.add((later, "fits"))
                        for l in range(32):
                            queue[l].append(sv[l])
                        continue
                    for l, v in enumerate(survivors(ch)):
                        queue[l].append(v)
                drain()
        except Undecided:
            return None
        return ev


def canon_rows(bank):
    """One id per distinct bank row (copies share it)."""
    return torch.unique(bank.view(torch.int16), dim=0, return_inverse=True)[1].numpy()


def warp_rows(X, mt, q, rows=256):
    """Image rows of warp q (0..7) of row tile mt; rows past B are zero (TMA fills them so)."""
    B, D = X.shape
    r0 = mt * rows + 32 * q
    x = torch.zeros(32, D, dtype=torch.bfloat16)
    n = max(0, min(32, B - r0))
    x[:n] = X[r0:r0 + n]
    return x


def reach(X, bank, canon, tiles_of_worker, KL, segs, warps=(0, 5)):
    """Union of the branches of the sampled warps of row tile 0 over the given segments (worker, first column)."""
    got, decided = set(), 0
    for w, a in segs:
        tiles = [t for t in tiles_of_worker(w) if t["mt"] == 0]
        tiles = next(sg for sg in segments(tiles) if sg[0]["col0"] == a)
        e = tiles[-1]["col0"] + tiles[-1]["nvalid"]
        for q in warps:
            ev = WarpModel(warp_rows(X, 0, q), bank[a:e], canon[a:e], KL).run(tiles, a)
            if ev is not None:
                decided += 1
                got |= ev
    return got, decided


def _worker_of(s, C, col):
    for w, a, e in row_tile_segments(s, C, 0):
        if a <= col < e:
            return w, a
    raise AssertionError(col)


def case_reach(name, kind):
    """{(entry point, variant, KL, later sub-tile, branch)} of one case, and the number of decided warps."""
    B, C, D, K = SHAPES[name]
    s = plan_sched(B, C, D, K)
    X, bank, info = case_inputs(name, kind)
    canon = canon_rows(bank)
    if kind == "tree":
        segs = [(w, a) for w, a, e in row_tile_segments(s, C, 0) if e - a >= RUN][:2]
    else:
        cols = [a for a, _ in info["runs"]] + info["tied"][:1]
        segs = sorted({_worker_of(s, C, c) for c in cols})
    lens = {("production", _ops().score_topk_plan(B, C, D, K)["list_len"]), ("exact", exact_len(K))}
    if name == "shard":
        lens.add(("scatter", _ops().global_list_len(B, C, D, K, SHARD_N * C)))
    out, n = set(), 0
    for variant, KL in sorted(lens):
        got, d = reach(X, bank, canon, lambda w: walk(s, C, w), KL, segs)
        n += d
        entry = "score_topk_scatter" if variant == "scatter" else "score_topk"
        out |= {(entry, "production" if variant == "scatter" else variant, KL, later, b) for later, b in got}
    return out, n


def splits_reach():
    B, C, D = SPLIT_SHAPE
    s = splits_sched()
    out, n = set(), 0
    for K in SPLIT_KS:
        X, bank, info = build_splits(K)
        canon = canon_rows(bank)
        walker = lambda w: walk_groups(s, SPLIT_ENDS, w)
        segs = [(w, a) for w, a, e in row_tile_segments(s, C, 0, walker)
                if any(a < re_ and ra < e for ra, re_ in info["runs"])]
        got, d = reach(X, bank, canon, walker, exact_len(K), segs)
        n += d
        out |= {("score_topk_splits", "exact", exact_len(K), later, b) for later, b in got}
    return out, n


def all_reach():
    out = set()
    for name, kinds in KINDS.items():
        for kind in kinds:
            got, n = case_reach(name, kind)
            assert n > 0 or kind == "tree", (name, kind, "no decided warp")
            out |= {(name, kind) + e for e in got}
    got, n = splits_reach()
    assert n > 0
    out |= {("splits", "rising") + e for e in got}
    return out


@pytest.fixture(scope="module")
def reached():
    r = all_reach()
    for e in sorted(r, key=str):
        print("reach", *e)
    return r


def _overflow(KL):
    return "fail_redo" if KL <= KC["drain_above"] else "early_drain"


def test_kernel_constants_are_read_from_the_sources():
    assert CHUNK < queue_len(8) <= queue_len(32) and SUB_N % UNIT == 0 and SUB_N % CHUNK == 0
    assert queue_len(KC["narrow"]) == KC["q_narrow"] and queue_len(KC["narrow"] + 2) == KC["q_wide"]


def test_every_list_length_overflows_its_queue_on_a_later_sub_tile(reached):
    """Rising runs: for production and for exact lists, every list length takes its overflow branch (a failed
    saturating append and its redo for the 56-entry queue, the early drain for the 64-entry one) on a sub-tile that is
    not the segment's first; the narrow queue also takes the saturating append that fits."""
    rising = {(entry, v, KL, b) for (_, kind, entry, v, KL, later, b) in reached if later and kind.startswith("rising")}
    for v, kls in (("production", (8, 10, 12, 16, 20, 32)), ("exact", (8, 12, 20, 32))):
        for KL in kls:
            assert ("score_topk", v, KL, _overflow(KL)) in rising, (v, KL)
            if KL <= KC["drain_above"]:
                assert ("score_topk", v, KL, "fits") in rising, (v, KL)
    assert ("score_topk_scatter", "production", 10, "fail_redo") in rising
    for KL in (exact_len(k) for k in SPLIT_KS):
        assert ("score_topk_splits", "exact", KL, _overflow(KL)) in rising, KL
    # the redo always fits: one chunk holds fewer survivors than the queue has slots
    assert all(b != "reload" for (*_, b) in reached)


def test_tied_runs_overflow_on_a_later_sub_tile(reached):
    """Copies of one row in a later sub-tile: the tie at the K-th value is cut across the overflow branch."""
    tied = {(name, v, KL, b) for (name, kind, _, v, KL, later, b) in reached if kind == "tied" and later}
    for name in (n for n, kinds in KINDS.items() if "tied" in kinds):
        B, C, D, K = SHAPES[name]
        for v, KL in (("production", _ops().score_topk_plan(B, C, D, K)["list_len"]), ("exact", exact_len(K))):
            assert (name, v, KL, _overflow(KL)) in tied, (name, v, KL)


def test_first_sub_tile_of_a_rising_run_does_not_overflow(reached):
    """The warm-up floor lets about KL values of a rising run through: only later sub-tiles overflow."""
    first = {b for (_, kind, *_, later, b) in reached if kind.startswith("rising") and not later}
    assert "fail_redo" not in first and "early_drain" not in first


def _lists(s, C, mt, walker=None):
    return [(a, e) for _, a, e in row_tile_segments(s, C, mt, walker)]


@pytest.mark.parametrize("name", [n for n, k in KINDS.items() if "rising_below_top" in k])
def test_rising_below_top_certifies_every_list(name):
    """Every full list of every row ends below the row's K-th value with margin (the list's KL-th largest upper bound
    below the K-th largest lower bound), so the production merge repairs nothing."""
    B, C, D, K = SHAPES[name]
    plan = _ops().score_topk_plan(B, C, D, K)
    KL = plan["list_len"]
    assert KL < K
    s = plan_sched(B, C, D, K)
    X, bank, info = case_inputs(name, "rising_below_top")
    x, w = X.double(), bank.double()
    lo_k = torch.empty(B, dtype=torch.float64)
    per_list = []
    for r0 in range(0, B, 256):
        xr = x[r0:r0 + 256]
        R = xr @ w.T
        E = (D + 2) * 2.0 ** -23 * (xr.abs() @ w.abs().T)
        lo_k[r0:r0 + 256] = (R - E).topk(K, 1).values[:, -1]
        worst = torch.full((xr.shape[0],), -float("inf"), dtype=torch.float64)
        for a, e in _lists(s, C, r0 // 256):
            if e - a >= KL:
                worst = torch.maximum(worst, (R + E)[:, a:e].topk(KL, 1).values[:, -1])
        per_list.append(worst)
        # the K top rows are the K largest values of every row, decided
        top_lo = (R - E)[:, info["top"]].min(1).values
        rest = torch.ones(C, dtype=torch.bool)
        rest[info["top"]] = False
        assert (top_lo > (R + E)[:, rest].max(1).values).all()
    assert (torch.cat(per_list) < lo_k).all()
    tops = torch.tensor(info["top"])
    for mt in range(s["MT"]):
        for a, e in _lists(s, C, mt):
            assert int(((tops >= a) & (tops < e)).sum()) < KL
