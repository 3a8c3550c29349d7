"""Kernel (2) bit for bit: every list length, merge kernel and schedule edge of the fused top-K against a sort of the
same GEMM's dense logits (``tests.util.reference_topk``), and the paths whose sums are not the tensor core's (``simt``,
rows repaired on the CUDA cores) against float64 (``tests.util.check_topk_f64``).

``GRID`` is built from ``ops.score_topk_plan`` and the constants of ``sched.cuh`` / ``umma_common.cuh``;
``tests/test_cpu_topk_grid.py`` checks without a GPU that it reaches every (list length, merge kernel) pair the policy
can produce, every remainder sub-tile width, both ring depths and both branches of ``pick_sched``."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from tests.util import _unit_bf16, check_topk_f64, reference_hits, reference_topk

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (B, C, D, K).  What each shape is for (production list length KL / merge kernel from the plan at 148 SMs):
GRID = [
    (512, 21841, 1024, 20),   # cfg 2: KL 8, 37 lists -> select<10>
    (2048, 300, 72, 20),      # ring depth 4 (B >= 2048), aligned pick_sched (72 workers, 8 row tiles)
    (9500, 20, 64, 20),       # 38 row tiles of 2 units: the sketch has solo and shared row tiles in one launch
    (2047, 1000, 64, 12),     # KL 10 speculative, rank<3>; ring depth 5; aligned branch
    (2047, 300, 64, 20),      # KL 16 speculative, select<6>
    (1, 300, 64, 13),         # KL 10 speculative, select<6>
    (1, 100, 64, 20),         # KL 16 speculative, select<4>
    (257, 4097, 1032, 21),    # unaligned pick_sched, KL 10 / merge<4>; D tail of 8 past 16 K blocks
    (2047, 1156, 56, 1),
    (2047, 2000, 8, 9),       # D = 8: one partial K block
    (2047, 4097, 64, 32),     # exact KL 32 with 9 lists
    (1, 1, 64, 7),
    (127, 1, 72, 12),
    (128, 50, 64, 13),
    (129, 71, 56, 16),
    (128, 300, 64, 7),
    (255, 197, 8, 8),
    (1, 1, 64, 21),
    (1, 36, 64, 21),
    (1, 50, 1032, 21),
    (1, 71, 64, 21),
    (1, 85, 64, 9),
    (1, 148, 72, 13),
    (1, 162, 64, 10),
    (1, 260, 64, 1),
    (1, 260, 56, 12),
    (1, 645, 64, 1),
    (1, 50, 64, 17),          # KL 16 speculative, rank<2>
    (1, 71, 64, 17),
    (1, 99, 8, 11),
    (1, 99, 64, 16),
    (1, 99, 64, 17),
    (1, 197, 64, 23),
    (1, 260, 72, 20),
    (1, 309, 64, 14),
    (1, 386, 64, 1),
    (1, 421, 64, 9),
    (1, 421, 1032, 28),
    (257, 596, 64, 30),
    (2047, 148, 64, 13),
    (1, 11866, 64, 20),       # remainder sub-tiles of 160 and 176 columns
    (255, 16602, 56, 12),     # remainder sub-tiles of 240 columns
]

# one production shape per merge kernel (rank<2>, rank<3>, select<4>, select<6>, select<10>, merge<4>), at least two
# lists per row, for the value-domain edges
EDGE_SHAPES = [(129, 48, 64, 13), (2047, 1000, 64, 12), (1, 100, 64, 20), (2047, 300, 64, 20), (1, 320, 64, 16),
               (257, 4097, 64, 21)]

SCALES = (1.0, 14.285714, 100.0)
IMPLS = ("tcgen05_exact", "tcgen05_sketch", "tcgen05", "simt")

ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from hgrnet_b200 import ops as _ops
    ops = _ops
    yield
    torch.cuda.synchronize()


def _impl(name):
    return {"simt": ops.HGR_IMPL_SIMT, "tcgen05": ops.HGR_IMPL_TCGEN05, "tcgen05_exact": ops.HGR_IMPL_TCGEN05_EXACT,
            "tcgen05_sketch": ops.HGR_IMPL_TCGEN05_SKETCH}[name]


def _rand(n, d, seed):
    return _unit_bf16(torch.randn(n, d, generator=torch.Generator().manual_seed(seed))).to(DEV)


def _poisoned(B, K, S=None):
    """Outputs every entry of which fails the comparison unless the kernel writes it."""
    shape = (B, K) if S is None else (S, B, K)
    return (torch.full(shape, float("nan"), device=DEV), torch.full(shape, 0x7FFFFFFF, dtype=torch.int32, device=DEV))


def _run(X, bank, K, impl, scale=1.0, col_id=None, id_base=0, targets=None):
    hits = ops.new_hits(DEV)
    out = _poisoned(X.shape[0], K)
    val, idx = ops.score_topk(X, bank, col_id=col_id, id_base=id_base, targets=targets, K=K, scale=scale, hits=hits,
                              impl=_impl(impl), out=out)
    assert val.data_ptr() == out[0].data_ptr()
    return val, idx, hits


def _check(impl, got_v, got_i, ref_v, ref_i, X, bank, K, scale, col_id=None, id_base=0):
    """tcgen05 variants: equal to the reference bit for bit; production: rows it re-scanned on the CUDA cores (at most
    ``last_rescan_count()`` of them) may differ and then pass the float64 check; ``simt``: the float64 check."""
    if impl == "simt":
        check_topk_f64(got_v, got_i, X, bank, K, scale, col_id, id_base)
        return
    rescans = ops.last_rescan_count(DEV) if impl == "tcgen05" else 0
    same = (got_v == ref_v).all(1) & (got_i == ref_i).all(1)
    bad = (~same).nonzero().flatten()
    assert bad.numel() <= rescans, "%s: %d rows differ from the reference (%d re-scanned), first row %d: %s %s vs %s %s" % (
        impl, bad.numel(), rescans, int(bad[0]), got_i[bad[0]].tolist(), got_v[bad[0]].tolist(), ref_i[bad[0]].tolist(),
        ref_v[bad[0]].tolist())
    check_topk_f64(got_v, got_i, X, bank, K, scale, col_id, id_base, rows=bad)


def _targets(B, col_id, id_base, C, seed):
    """Ids of random bank rows, with -1 (padding) and ids of no bank row mixed in."""
    g = torch.Generator().manual_seed(seed)
    rows = torch.randint(0, C, (B,), generator=g)
    t = (col_id.cpu()[rows].long() if col_id is not None else rows + id_base).int()
    t[::7] = -1
    t[3::11] = (int(col_id.max()) + 5) if col_id is not None else id_base + C + 5
    return t.to(DEV)


@pytest.mark.parametrize("B,C,D,K", GRID)
def test_single_bank_topk_is_the_sorted_dense_logits(B, C, D, K):
    """Every variant on every grid shape: exact and sketch equal the reference on every row, production too unless it
    re-scanned rows, simt within the float64 bound; the hit counters are those of the returned ids."""
    i = GRID.index((B, C, D, K))
    scale = SCALES[i % 3]
    X, bank = _rand(B, D, 100 + i), _rand(C, D, 200 + i)
    if i % 2:
        col_id, id_base = None, 1000 + i
    else:
        col_id, id_base = torch.from_numpy(np.random.RandomState(i).permutation(10 * C)[:C].astype(np.int32)).to(DEV), 0
    targets = _targets(B, col_id, id_base, C, i)
    ref_v, ref_i = reference_topk(X, bank, K, scale, col_id, id_base)
    for impl in IMPLS:
        if impl == "tcgen05_sketch" and K > 20:
            continue
        val, idx, hits = _run(X, bank, K, impl, scale, col_id, id_base, targets)
        _check(impl, val, idx, ref_v, ref_i, X, bank, K, scale, col_id, id_base)
        assert hits.tolist() == reference_hits(idx, targets), impl
        if impl != "simt" and impl != "tcgen05":
            assert hits.tolist() == reference_hits(ref_i, targets), impl


def _edge_bank(C, D, K, cpw, seed):
    """Bank with two anchor rows copied exactly to chosen places, a few zero rows, the rest random.  Anchor A sits at
    the first and last column, on both sides of every worker-chunk boundary (multiples of ``cpw``) and of every
    sub-tile boundary (multiples of 256 inside a chunk), as a run of 40 rows from the second chunk's first column (so a
    first sub-tile is filled with it: the warm-up floor equals the anchor's value) and at further rows until there are
    K + 3 copies: the cut falls inside the ties.  Anchor B takes half as many places, so its ties are ordered inside the
    list.  Every row leans on one direction u (``-u`` is anti-aligned with the whole bank)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(D, generator=g)
    u = u / u.norm()
    bank = _unit_bf16(torch.randn(C, D, generator=g) + 8.0 * u).to(DEV)
    pos = {0, C - 1}
    for b in range(cpw, C, cpw):
        pos |= {b - 1, b}
    for c0 in range(0, C, cpw):
        for s in range(c0 + 256, min(c0 + cpw, C), 256):
            pos |= {s - 1, s}
    if cpw < C:
        pos |= set(range(cpw, min(cpw + 40, C)))
    rest = [r for r in range(1, C - 1) if r not in pos]
    extra = max(0, K + 3 - len(pos))
    pos |= set(rest[:: max(1, len(rest) // max(extra, 1))][:extra])
    pos_a = sorted(pos)
    free = [r for r in range(C) if r not in pos]
    pos_b = free[1::max(1, len(free) // max(K // 2, 1))][:max(K // 2, 1)]
    zeros = [r for r in free[::7] if r not in pos_b][:5]
    bank[pos_a] = bank[pos_a[0]].clone()
    bank[pos_b] = bank[pos_b[0]].clone()
    bank[zeros] = 0
    return bank, pos_a, pos_b, u.to(DEV)


def _edge_queries(B, bank, pos_a, pos_b, u, seed):
    """Rows near anchor A, near anchor B, and anti-aligned with the bank (every logit negative but those of the zero
    rows)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    D = bank.shape[1]
    a, b = bank[pos_a[0]].float(), bank[pos_b[0]].float()
    noise = 0.05 * torch.randn(B, D, device=DEV, generator=g)
    kind = torch.arange(B, device=DEV) % 3
    x = torch.where((kind == 0)[:, None], a + noise, torch.where((kind == 1)[:, None], b + noise, -u + 0.4 * noise))
    return _unit_bf16(x)


@pytest.mark.parametrize("B,C,D,K", EDGE_SHAPES)
def test_value_edges_reach_every_merge_kernel(B, C, D, K):
    """Exact ties across worker-chunk and sub-tile boundaries, at the first and last column and at the K-th position
    (they resolve by ascending bank row), queries anti-aligned with the bank, zero bank rows, three scales; and with
    K = 32 on exact lists.  The zero rows meet queries of mixed signs, so their logits are +0 (no -0 enters a list)."""
    plan = ops.score_topk_plan(B, C, D, K)
    bank, pos_a, pos_b, u = _edge_bank(C, D, K, plan["cols_per_worker"], seed=C)
    X = _edge_queries(B, bank, pos_a, pos_b, u, seed=B)
    zero = (bank == 0).all(1)
    assert ((X[2::3].float() @ bank[~zero].float().T) < 0).all()
    for scale in SCALES:
        for k, impls in ((K, IMPLS), (32, ("tcgen05_exact", "simt"))):
            ref_v, ref_i = reference_topk(X, bank, k, scale)
            for impl in impls:
                if impl == "tcgen05_sketch" and k > 20:
                    continue
                val, idx, _ = _run(X, bank, k, impl, scale)
                _check(impl, val, idx, ref_v, ref_i, X, bank, k, scale)


@pytest.mark.parametrize("K", [1, 7, 13, 20, 32])
def test_fewer_classes_than_and_around_K(K):
    """C in {1, K - 1, K, K + 1}: lists padded with (-inf, -1) exactly when C < K."""
    for C in sorted({1, max(K - 1, 1), K, K + 1}):
        X, bank = _rand(33, 64, K), _rand(C, 64, K + C)
        ref_v, ref_i = reference_topk(X, bank, K, 14.285714)
        for impl in IMPLS:
            if impl == "tcgen05_sketch" and K > 20:
                continue
            val, idx, _ = _run(X, bank, K, impl, 14.285714)
            _check(impl, val, idx, ref_v, ref_i, X, bank, K, 14.285714)


@pytest.mark.parametrize("B,C,K,KL", [(129, 300, 12, 8), (129, 200, 13, 10), (129, 200, 20, 12), (129, 200, 32, 16),
                                      (255, 5000, 20, 8)])
def test_speculative_lists_repaired_at_every_list_length(B, C, K, KL):
    """Near-copies of the mean query direction inside one worker's chunk (the queries are spread around one direction,
    so the copies lead every row) overflow that worker's speculative lists: the rows are re-scanned on the CUDA cores
    and pass the float64 check; the other rows equal the reference."""
    D = 64
    plan = ops.score_topk_plan(B, C, D, K)
    assert plan["list_len"] == KL
    cpw = plan["cols_per_worker"]
    g = torch.Generator().manual_seed(7)
    X = _unit_bf16(torch.randn(1, D, generator=g) + 0.5 * torch.randn(B, D, generator=g) / D ** 0.5).to(DEV)
    bank = _rand(C, D, 8).clone()
    mean = X.float().mean(0)
    mean = mean / mean.norm()
    r0 = (C // 2) // cpw * cpw
    n = min(cpw, 40)
    bank[r0:r0 + n] = _unit_bf16(3 * mean[None, :].cpu() + torch.randn(n, D, generator=torch.Generator().manual_seed(9))
                                 / D ** 0.5).to(DEV)
    ref_v, ref_i = reference_topk(X, bank, K)
    val, idx, _ = _run(X, bank, K, "tcgen05")
    assert ops.last_rescan_count(DEV) > 0, "the adversarial bank should overflow speculative lists"
    _check("tcgen05", val, idx, ref_v, ref_i, X, bank, K, 1.0)
    check_topk_f64(val, idx, X, bank, K)


@pytest.mark.parametrize("kind", ["iid", "clustered"])
def test_global_certificate_bound_is_sound(kind):
    """``score_topk_scatter`` with bounds (one class shard of a row's global stream, lists sized for the owner's
    certificate): per row, every emitted entry above the bound is the shard's reference entry at that position, and no
    bank row left out beats the emitted K-th entry in (value desc, row asc) unless its value is <= the bound."""
    from tests.util import hostile_bank, hostile_queries
    B, C, D, K = 1024, 2731, 256, 32
    bank = hostile_bank(C, D, kind).to(DEV)
    X = hostile_queries(bank, B, kind)
    ref_v, ref_i = reference_topk(X, bank, C)           # every column, sorted: ranks of all bank rows
    acc = ops.logits_dense(X, bank)
    seen = set()
    for C_total in (C, 2 * C, 4 * C, 8 * C):
        KL = ops.global_list_len(B, C, D, K, C_total)
        seen.add(KL)
        blocks = 2
        br = (B + blocks - 1) // blocks
        vals = [torch.full((br, K), float("nan"), device=DEV) for _ in range(blocks)]
        idxs = [torch.full((br, K), 0x7FFFFFFF, dtype=torch.int32, device=DEV) for _ in range(blocks)]
        bnds = [torch.full((br,), float("nan"), device=DEV) for _ in range(blocks)]
        ops.score_topk_scatter(X, bank, [v.data_ptr() for v in vals], [i.data_ptr() for i in idxs], br, K=K,
                               bound_block_ptrs=[b.data_ptr() for b in bnds], C_total=C_total)
        v, i, bound = torch.cat(vals)[:B], torch.cat(idxs)[:B].long(), torch.cat(bnds)[:B]
        assert not torch.isnan(bound).any() and not torch.isnan(v).any()
        above = v > bound[:, None]
        assert torch.equal(torch.where(above, v, 0.0), torch.where(above, ref_v[:, :K], 0.0)), (kind, C_total, KL)
        assert torch.equal(torch.where(above, i, 0), torch.where(above, ref_i[:, :K].long(), 0)), (kind, C_total, KL)
        # rank of every bank row in the reference order; the emitted K-th entry's rank
        rank = torch.empty_like(ref_i, dtype=torch.long).scatter_(1, ref_i.long(), torch.arange(C, device=DEV).expand(B, C))
        emitted = torch.zeros(B, C, dtype=torch.bool, device=DEV).scatter_(1, i.clamp_min(0), i >= 0)
        kth = torch.where(i[:, -1] >= 0, rank.gather(1, i[:, -1:].clamp_min(0)).squeeze(1), torch.full_like(i[:, -1], C))
        beats = ~emitted & (rank < kth[:, None]) & (acc > bound[:, None])
        assert not beats.any(), (kind, C_total, KL, int(beats.any(1).sum()))
    assert seen >= {8, 10, 12, 16}, seen


@pytest.mark.parametrize("K", [13, 32])
@pytest.mark.parametrize("impl", ["tcgen05", "tcgen05_exact"])
def test_splits_equal_the_reference_of_each_split(K, impl):
    """Groups of 1, 15, 17, 255 and 257 rows (units start at unaligned bank rows): split s equals the reference over
    its union-bank rows, bit for bit (production: rows it re-scanned pass the float64 check)."""
    sizes = [1, 15, 17, 255, 257, 33]
    masks = [0b01, 0b10, 0b11, 0b01, 0b11, 0b10]
    ends = np.cumsum(sizes).tolist()
    C, B, D = ends[-1], 300, 72
    X, bank = _rand(B, D, 31), _rand(C, D, 32)
    col_id = torch.from_numpy(np.random.RandomState(3).permutation(5 * C)[:C].astype(np.int32)).to(DEV)
    out = _poisoned(B, K, 2)
    val, idx = ops.score_topk_splits(X, bank, ends, masks, 2, col_id=col_id, K=K, scale=14.285714, impl=_impl(impl),
                                     out=out)
    rescans = ops.last_rescan_count(DEV)
    starts = [0] + ends[:-1]
    for s in range(2):
        rows = torch.cat([torch.arange(a, e) for a, e, m in zip(starts, ends, masks) if (m >> s) & 1]).to(DEV)
        ref_v, ref_i = reference_topk(X, bank[rows].contiguous(), K, 14.285714, col_id[rows])
        sub = bank[rows].contiguous()
        same = (val[s] == ref_v).all(1) & (idx[s] == ref_i).all(1)
        bad = (~same).nonzero().flatten()
        assert bad.numel() <= (rescans if impl == "tcgen05" else 0), (s, bad.numel(), rescans)
        check_topk_f64(val[s], idx[s], X, sub, K, 14.285714, col_id[rows], rows=bad)


# level sizes: boundaries at 15 / 16 / 17 and 255 / 256 / 257 columns, one-column levels, and level 3 without train rows
_LEVEL_SIZES = (15, 1, 1, 0, 238, 1, 1, 300, 1)


@pytest.mark.parametrize("B,D", [(1, 64), (127, 72), (129, 8), (257, 1032)])
def test_level_argmax_ties_at_level_and_tile_edges(B, D):
    """``hier_metrics_fused_rows``: per-level winners against ``oracle.tor_por_winners`` on the dense logits of the same
    GEMM.  One bank row is copied into every level, and half the image rows lie near it, so each level's maximum is an
    exact tie and the first position must win.  In a short level the copies are its first, fifth, 33rd and 37th row and
    its last row: ties across the level boundaries, chunks and sub-tiles.  In a long level they start at a row 1 mod 16
    at least 40 rows in: the first two copies then share a 32-column chunk that lies inside the level (a chunk starts
    at a multiple of 16) and the same one of its four running maxima, with no earlier copy to hide the tie-break there.
    A level without train rows takes the first position (its masked array is all -1)."""
    from hgrnet_b200.evaluate import chain_table
    from oracle import hgr_oracle as orc
    level_of, train = [], []
    for l, n in enumerate(_LEVEL_SIZES):
        level_of += [l] * max(n, 1)                   # an empty level still has a (non-train) node
        train += [True] * n + [False] * (n == 0)
    N = len(level_of)
    train_index = torch.tensor([n for n in range(N) if train[n]])
    M = len(train_index)
    first = {l: level_of.index(l) for l in range(len(_LEVEL_SIZES))}
    c2p = [[first[j] for j in range(level_of[n])] for n in range(N)]
    d2n = {l: [n for n in range(N) if level_of[n] == l] for l in range(len(_LEVEL_SIZES))}
    depth = np.asarray(level_of)
    bank = _rand(M, D, 41).clone()
    ends = np.cumsum(_LEVEL_SIZES).tolist()
    for s, e in zip([0] + ends[:-1], ends):
        p = s if e - s < 128 else s + 40 + (1 - (s + 40)) % 16
        copies = [c for c in (p, p + 4, p + 32, p + 36, e - 1) if s <= c < e]
        bank[copies] = bank[0].clone()
    g = torch.Generator(device=DEV).manual_seed(D)
    x = torch.randn(B, D, device=DEV, generator=g)
    x[::2] = bank[0].float() + 0.05 * x[::2]
    x = _unit_bf16(x)
    dt = torch.tensor(level_of)[train_index]
    first_out = torch.tensor([int((dt != l).nonzero()[0]) if (dt != l).any() else M for l in range(len(_LEVEL_SIZES))],
                             dtype=torch.int32, device=DEV)
    table = [torch.from_numpy(a).to(DEV) for a in chain_table(c2p, depth, train_index.tolist())]
    lvl = torch.full((B, len(_LEVEL_SIZES)), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
    top1 = torch.full((B,), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
    target = N - 1
    ops.hier_metrics_fused_rows(x, bank, ends, torch.arange(M, dtype=torch.int32, device=DEV), first_out,
                                torch.full((B,), target, dtype=torch.int32, device=DEV), *table,
                                ops.new_hier_counts(DEV), lvl_idx=lvl, top1=top1)
    logits = torch.zeros(B, N)
    logits[:, train_index] = ops.logits_dense(x, bank).cpu()
    top1_ref, path = orc.tor_por_winners(logits, train_index, c2p, d2n, N, target)
    assert torch.equal(train_index[lvl.cpu().long()], path), "per-level winners differ"
    assert torch.equal(train_index[top1.cpu().long()], top1_ref), "top-1 differs"
