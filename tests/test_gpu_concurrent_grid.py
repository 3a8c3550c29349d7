"""The scoring kernel on a share of the grid (``ops.score_topk(grid_share=c)``, ``HGR_IMPL_GRID_SHARE``) computes what
it computes on the whole grid.

A share only re-cuts the bank columns among fewer CTA pairs: longer worker ranges, fewer and longer lists per row, and
with them other list lengths and merge kernels.  A logit does not depend on its column's place in a tile and ties are
ordered by (value desc, bank row asc) however the lists are cut, so ``tcgen05_exact`` must equal the sort of the same
GEMM's dense logits (``tests.util.reference_topk``) bit for bit at every share, and the production kernel too on every
row it did not repair.  Hostile banks make the production kernel repair, on the longer list ranges of a share.  Two
streams at different shares run at the same time into one counter buffer, and the plan ``EvalStream`` picks at cfg 2
leaves room for a normalise and a merge CTA beside its scoring CTA."""
from __future__ import annotations

import numpy as np
import pytest
import torch

import tests.test_gpu_topk_exact as exact_tests
from tests.test_gpu_colocation import _device_limits, _regs, _smem
from tests.test_gpu_topk_exact import _check, _impl, _poisoned, _rand, _targets
from tests.util import hostile_bank, hostile_queries, reference_hits, reference_topk

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHARES = (1, 2, 3, 4)

# (B, C, D, K): cfg 2, cfg 4, and ragged shapes (row tiles of 1 and 257 rows, C off the 16-row unit, D tails)
SHAPES = [
    (512, 21841, 1024, 20),
    (1024, 10450, 512, 20),
    (257, 4097, 1032, 21),
    (700, 2731, 72, 20),
    (1, 300, 64, 13),
    (1999, 5003, 56, 12),
]
HOSTILE = ("clustered", "equal", "dups")

ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from hgrnet_b200 import ops as _ops
    ops = _ops
    exact_tests.ops = _ops          # _check reads the module global of its own file
    yield
    torch.cuda.synchronize()


def _run(X, bank, K, impl, share, col_id=None, id_base=0, targets=None, hits=None):
    hits = ops.new_hits(DEV) if hits is None else hits
    val, idx = ops.score_topk(X, bank, col_id=col_id, id_base=id_base, targets=targets, K=K, hits=hits,
                              impl=_impl(impl), out=_poisoned(X.shape[0], K), grid_share=share)
    return val, idx, hits


@pytest.mark.parametrize("B,C,D,K", SHAPES)
def test_every_share_equals_the_sorted_dense_logits_and_the_full_grid(B, C, D, K):
    i = SHAPES.index((B, C, D, K))
    X, bank = _rand(B, D, 300 + i), _rand(C, D, 400 + i)
    col_id = torch.from_numpy(np.random.RandomState(i).permutation(3 * C)[:C].astype(np.int32)).to(DEV)
    targets = _targets(B, col_id, 0, C, i)
    ref_v, ref_i = reference_topk(X, bank, K, 1.0, col_id)
    full = {}
    for share in SHARES:
        for impl in ("tcgen05_exact", "tcgen05"):
            val, idx, hits = _run(X, bank, K, impl, share, col_id, targets=targets)
            if impl == "tcgen05_exact":
                assert torch.equal(val, ref_v) and torch.equal(idx, ref_i), share
                assert hits.tolist() == reference_hits(ref_i, targets), share
                continue
            rescans = ops.last_rescan_count(DEV)
            _check(impl, val, idx, ref_v, ref_i, X, bank, K, 1.0, col_id)
            assert hits.tolist() == reference_hits(idx, targets), share
            if share == 1:
                full = dict(val=val, idx=idx, rescans=rescans)
            elif rescans == 0 and full["rescans"] == 0:
                assert torch.equal(val, full["val"]) and torch.equal(idx, full["idx"]), share


@pytest.mark.parametrize("kind", HOSTILE)
@pytest.mark.parametrize("B,C,D,K", [(512, 8191, 64, 20), (300, 3001, 128, 12)])
def test_every_share_on_hostile_banks(kind, B, C, D, K):
    """Banks whose row order is not random: the production kernel's lists fail to certify and the merge repairs them
    over the share's longer column ranges; the result is still exact."""
    bank = hostile_bank(C, D, kind).to(DEV)
    X = hostile_queries(bank, B, kind)
    targets = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(C)).int().to(DEV)
    ref_v, ref_i = reference_topk(X, bank, K)
    for share in SHARES:
        val, idx, hits = _run(X, bank, K, "tcgen05_exact", share, targets=targets)
        assert torch.equal(val, ref_v) and torch.equal(idx, ref_i), share
        val, idx, hits = _run(X, bank, K, "tcgen05", share, targets=targets)
        _check("tcgen05", val, idx, ref_v, ref_i, X, bank, K, 1.0)
        assert hits.tolist() == reference_hits(idx, targets), share


def test_two_streams_at_different_shares_count_into_one_buffer():
    B, C, D, K = 512, 21841, 1024, 20
    X = [_rand(B, D, 500 + s) for s in range(2)]
    bank = _rand(C, D, 600)
    targets = [_targets(B, None, 0, C, 700 + s) for s in range(2)]
    refs = [reference_topk(X[s], bank, K) for s in range(2)]
    hits = ops.new_hits(DEV)
    streams = [torch.cuda.Stream() for _ in range(2)]
    out = [None, None]
    cur = torch.cuda.current_stream()
    for share_a, share_b in ((2, 3), (1, 4), (2, 2)):
        hits.zero_()
        for st in streams:
            st.wait_stream(cur)
        for rep in range(4):
            for s, (st, share) in enumerate(zip(streams, (share_a, share_b))):
                with torch.cuda.stream(st):
                    out[s] = ops.score_topk(X[s], bank, targets=targets[s], K=K, hits=hits,
                                            impl=ops.HGR_IMPL_TCGEN05_EXACT, grid_share=share)
        for st in streams:
            cur.wait_stream(st)
        torch.cuda.synchronize()
        want = [0] * ops.HGR_NUM_HITS
        for s in range(2):
            assert torch.equal(out[s][0], refs[s][0]) and torch.equal(out[s][1], refs[s][1]), (share_a, share_b, s)
            want = [w + 4 * h for w, h in zip(want, reference_hits(refs[s][1], targets[s]))]
        assert hits.tolist() == want, (share_a, share_b)


def test_eval_stream_runs_the_recommended_share_with_the_results_of_the_full_grid():
    """``EvalStream`` at cfg 2 on several streams picks the library's share (its plan: 36 pairs, 18 lists of 10 per
    row) and its counters and lists equal those of ``concurrent=1``."""
    from hgrnet_b200.stream import EvalStream
    B, C, D, K = 512, 21841, 1024, 20
    bank = _rand(C, D, 800)
    feats = [torch.randn(B, D, generator=torch.Generator().manual_seed(900 + s)).to(DEV) for s in range(4)]
    labels = [_targets(B, None, 0, C, 950 + s) for s in range(4)]
    runs = {}
    for concurrent in (None, 1):
        es = EvalStream(bank, batch=B, K=K, slots=4, streams=4, host_io=False, concurrent=concurrent)
        for s in range(4):
            es.dev_feats[s].copy_(feats[s])
            es.dev_labels[s].copy_(labels[s])
        es.begin()
        for i in range(8):
            es.step(i % 4)
        es.end()
        torch.cuda.synchronize()
        runs[concurrent] = (es.plan(), es.hit_counts(), [v.clone() for v in es.val], [x.clone() for x in es.idx])
    plan, hits, val, idx = runs[None]
    assert plan["grid_share"] == ops.score_topk_grid_share(B, C, D, K) == 2
    assert (plan["workers"], plan["lists_per_row"], plan["list_len"]) == (36, 18, 10)
    assert runs[1][0]["grid_share"] == 1 and runs[1][0]["workers"] == 74
    assert hits == runs[1][1]
    for s in range(4):
        assert torch.equal(val[s], runs[1][2][s]) and torch.equal(idx[s], runs[1][3][s]), s


@pytest.mark.parametrize("x_dtype", [torch.bfloat16, torch.float32])
def test_normalise_and_merge_fit_beside_the_scoring_cta_of_the_eval_stream_plan(x_dtype):
    """The list length of the share ``EvalStream`` runs at cfg 2 selects another scoring kernel instantiation: one CTA
    of it, one of the normalise and two of the merge still fit on one SM in shared memory, and the scoring CTA, a
    normalise and a merge CTA in registers (the rule of ``tests/test_gpu_colocation.py``)."""
    B, C, D, K = 512, 21841, 1024, 20
    share = ops.score_topk_grid_share(B, C, D, K)
    lim = _device_limits()
    fp = ops.score_topk_footprint(B, C, D, K, x_dtype=x_dtype, grid_share=share)
    smem = sum(_smem(f, lim["reserved_smem_per_block"]) for f in (fp["score"], fp["normalize"], fp["merge"], fp["merge"]))
    regs = sum(_regs(f) for f in (fp["score"], fp["normalize"], fp["merge"]))
    assert smem <= lim["smem_per_sm"], (smem, lim, fp)
    assert regs <= lim["regs_per_sm"], (regs, lim, fp)
