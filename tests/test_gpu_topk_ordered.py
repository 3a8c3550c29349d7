"""The top-K epilogues bit for bit on ordered banks whose runs overflow the candidate queues.

The inputs are built on the host (``tests/test_cpu_topk_ordered.py``), where a float64 restatement of the epilogue
shows which queue branch each case takes: every list length takes its overflow branch -- the failed saturating append
and its redo, or the early drain -- on a later sub-tile, and copies of one row cut the tie at the K-th value across it.
Here the kernels run on the same inputs: ``tcgen05_exact`` and ``tcgen05_sketch`` must equal the sort of the same GEMM's
logits (``tests.util.reference_topk``) on every row; the production kernel must repair nothing where every list
certifies, and elsewhere differ only on rows it repaired, which pass the float64 check."""
from __future__ import annotations

import pytest
import torch

import tests.test_gpu_topk_exact as exact_tests
from tests.test_cpu_topk_ordered import (KINDS, SHAPES, SHARD_N, SPLIT_ENDS, SPLIT_KS, SPLIT_MASKS, SPLIT_SHAPE,
                                         build_shard, build_splits, case_inputs)
from tests.test_gpu_topk_exact import _check, _impl, _poisoned, _run
from tests.util import check_topk_f64, reference_hits, reference_topk

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SCALES = (1.0, 14.285714)
ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from hgrnet_b200 import ops as _ops
    ops = _ops
    exact_tests.ops = _ops          # _run / _check read the module global of their own file
    yield
    torch.cuda.synchronize()


def _targets(B, C, seed):
    t = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(seed)).int()
    t[::5] = -1
    return t.to(DEV)


CASES = [(name, kind) for name, kinds in KINDS.items() for kind in kinds]


@pytest.mark.parametrize("name,kind", CASES)
def test_ordered_bank_equals_the_reference(name, kind):
    B, C, D, K = SHAPES[name]
    X, bank, info = case_inputs(name, kind)
    X, bank = X.to(DEV), bank.to(DEV)
    targets = _targets(B, C, B + C)
    for scale in SCALES:
        ref_v, ref_i = reference_topk(X, bank, K, scale)
        if kind == "tied":
            # the K-th entry of every row is the first copy of the tied row
            assert (ref_i[:, K - 1] == info["tied"][0]).all()
        for impl in ("tcgen05_exact", "tcgen05_sketch"):
            if impl == "tcgen05_sketch" and K > 20:
                continue
            val, idx, hits = _run(X, bank, K, impl, scale, targets=targets)
            assert torch.equal(val, ref_v) and torch.equal(idx, ref_i), (impl, scale, int(
                ((val != ref_v).any(1) | (idx != ref_i).any(1)).sum()))
            assert hits.tolist() == reference_hits(ref_i, targets), impl
        # production: a whole repaired cfg-2 tree bank costs about a second; there the exact lists above suffice
        if kind == "tree" and name.startswith("cfg2"):
            continue
        val, idx, hits = _run(X, bank, K, "tcgen05", scale, targets=targets)
        if kind == "rising_below_top":
            assert ops.last_rescan_count(DEV) == 0, "a list lost a candidate or failed to certify"
            assert torch.equal(val, ref_v) and torch.equal(idx, ref_i)
        else:
            _check("tcgen05", val, idx, ref_v, ref_i, X, bank, K, scale)
        assert hits.tolist() == reference_hits(idx, targets)


@pytest.mark.parametrize("K", SPLIT_KS)
@pytest.mark.parametrize("impl", ["tcgen05_exact", "tcgen05"])
def test_grouped_epilogue_on_runs_across_and_filling_groups(K, impl):
    """``score_topk_splits``: a rising run crosses the end of group 0, another fills group 2; each split equals the
    reference over its rows (production: rows it re-scanned pass the float64 check)."""
    X, bank, _ = build_splits(K)
    X, bank = X.to(DEV), bank.to(DEV)
    B, C, D = SPLIT_SHAPE
    starts = [0] + SPLIT_ENDS[:-1]
    for scale in SCALES:
        out = _poisoned(B, K, 2)
        val, idx = ops.score_topk_splits(X, bank, SPLIT_ENDS, SPLIT_MASKS, 2, K=K, scale=scale, impl=_impl(impl), out=out)
        rescans = ops.last_rescan_count(DEV) if impl == "tcgen05" else 0
        for s in range(2):
            rows = torch.cat([torch.arange(a, e) for a, e, m in zip(starts, SPLIT_ENDS, SPLIT_MASKS) if (m >> s) & 1])
            rows = rows.to(DEV)
            sub = bank[rows].contiguous()
            ref_v, ref_i = reference_topk(X, sub, K, scale, rows.int())
            bad = (~((val[s] == ref_v).all(1) & (idx[s] == ref_i).all(1))).nonzero().flatten()
            assert bad.numel() <= rescans, (impl, scale, s, bad.numel(), rescans)
            check_topk_f64(val[s], idx[s], X, sub, K, scale, rows.int(), rows=bad)


def test_class_shard_producer_on_a_rising_shard():
    """``score_topk_scatter`` with bounds for one shard of eight (global list length 10): every entry above the bound
    is the shard's reference entry, and no left-out bank row beats the K-th entry unless it is at or below the bound."""
    B, C, D, K = SHAPES["shard"]
    X, bank, _ = build_shard()
    X, bank = X.to(DEV), bank.to(DEV)
    C_total = SHARD_N * C
    assert ops.global_list_len(B, C, D, K, C_total) == 10
    ref_v, ref_i = reference_topk(X, bank, C)
    acc = ops.logits_dense(X, bank)
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
    assert above[:, 0].any(), "no row has an entry above its bound: the test would check nothing"
    assert torch.equal(torch.where(above, v, 0.0), torch.where(above, ref_v[:, :K], 0.0))
    assert torch.equal(torch.where(above, i, 0), torch.where(above, ref_i[:, :K].long(), 0))
    rank = torch.empty_like(ref_i, dtype=torch.long).scatter_(1, ref_i.long(), torch.arange(C, device=DEV).expand(B, C))
    emitted = torch.zeros(B, C, dtype=torch.bool, device=DEV).scatter_(1, i.clamp_min(0), i >= 0)
    kth = torch.where(i[:, -1] >= 0, rank.gather(1, i[:, -1:].clamp_min(0)).squeeze(1), torch.full_like(i[:, -1], C))
    beats = ~emitted & (rank < kth[:, None]) & (acc > bound[:, None])
    assert not beats.any(), int(beats.any(1).sum())
