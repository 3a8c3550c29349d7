"""TOR / POR with one label per row (``hgr_hier_metrics_fused_rows``, main.py:143,152-191) against the oracle's
restatement of the reference, directly and through ``HierMetrics.update_rows``, and inside the graph-replayed
``EvalStream``."""
from __future__ import annotations

import ctypes
import types

import pytest
import torch

from oracle import cases, hgr_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _emb(n, d, seed, normalize=True):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    if normalize:
        x = x / x.norm(dim=-1, keepdim=True)
    return x.to(torch.bfloat16).float()


def _setup(levels, B, D, train_every):
    """Seeded inputs with exact ties from duplicated bank rows (inside a level and across two levels), the arguments of
    ``hier_metrics_fused_rows``, the chain table and the train rows of the bank in ``train_index`` order."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import chain_table
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    h = synthetic_hierarchy(list(levels), seed=3)
    N = len(h)
    bank = _emb(N, D, 21).to(torch.bfloat16)
    bank[5] = bank[3]
    bank[N - 2] = bank[N // 2]
    if N > 7:
        bank[7] = bank[N - 1]                                   # a tie across two levels
    x = ops.normalize_rows(_emb(B, D, 22, normalize=False).to(DEV))
    train_index = torch.arange(0, N, train_every)
    depth = torch.from_numpy(h.depth).long()
    n_levels = int(depth.max()) + 1
    dt = depth[train_index]
    M = len(train_index)
    first_out = torch.tensor([int((dt != l).nonzero()[0]) if (dt != l).any() else M for l in range(n_levels)],
                             dtype=torch.int32, device=DEV)
    order = torch.sort(dt, stable=True).indices
    bank_train = bank[train_index].to(DEV).contiguous()
    args = dict(bank_sorted=bank_train[order.to(DEV)].contiguous(),
                level_end=torch.cumsum(torch.bincount(dt, minlength=n_levels), 0).tolist(),
                sorted_to_pos=order.to(torch.int32).to(DEV), first_out=first_out)
    table = [torch.from_numpy(a).to(DEV) for a in chain_table(h.c2p, h.depth, train_index.tolist())]
    return h, x, train_index, n_levels, args, dict(zip(("chain_ptr", "chain_pos", "chain_level"), table)), bank_train


def _oracle_logits(x, bank_train, train_index, n_nodes):
    """The fp32 logits of the fused GEMM (bit-identical to ``hgr_logits_dense`` on the same inputs) at the train columns
    of a ``[B, n_nodes]`` matrix; ``oracle.tor_por`` reads no other column."""
    from hgrnet_b200 import ops
    logits = torch.zeros(x.shape[0], n_nodes)
    logits[:, train_index] = ops.logits_dense(x, bank_train).cpu()
    return logits


def _oracle_bin(logits, train_index, h, target):
    """``oracle.tor_por`` of a single-label batch as the integers of bin L: ``[rows, TOR hits, points, edges]``."""
    tor, path_add, point_add = orc.tor_por(logits, train_index, h.c2p, h.d2n, len(h), target)
    L = len(h.c2p[target]) + 1
    return torch.tensor([logits.shape[0], int(tor), round(point_add * L), round(path_add * max(L - 1, 1))])


def _check_winners(logits, train_index, h, lvl, top1):
    """Per-level winners and top-1 (train positions) against the oracle's arg-maxes; the chain of the last node (the
    deepest level) covers every level."""
    _, dict_path = orc.tor_por_winners(logits, train_index, h.c2p, h.d2n, len(h), len(h) - 1)
    assert dict_path.shape[1] == lvl.shape[1]
    assert torch.equal(train_index[lvl.cpu().long()], dict_path), "per-level winners differ"
    assert torch.equal(train_index[top1.cpu().long()], train_index[logits[:, train_index].argmax(1)]), \
        "top-1 over the train classes differs"


_LEVELS6 = (6, 60, 600, 2400, 1500, 400)
_LEVELS12 = (20, 150, 900, 3000, 5500, 5500, 3500, 1800, 900, 400, 120, 51)      # cfg 2: 21,841 nodes, 12 levels
_LEVELS20 = tuple(1 + i // 2 for i in range(20))


@pytest.mark.parametrize("levels,B,D,train_every", [((4, 20, 200), 64, 64, 1), ((4, 20, 200), 64, 128, 1),
                                                    ((3, 9, 40, 160), 33, 64, 2), ((3, 9, 40, 160), 33, 128, 2),
                                                    ((1, 5), 7, 64, 1), (_LEVELS20, 9, 64, 1), (_LEVELS20, 9, 128, 1),
                                                    (_LEVELS6, 12, 128, 1), (_LEVELS6, 5, 64, 3),
                                                    (_LEVELS6, 300, 256, 1), (_LEVELS12, 512, 1024, 1)])
def test_hier_rows_match_oracle(levels, B, D, train_every):
    """Single-label batches: bin L of the counters, the per-level winners and the top-1 equal the oracle's on the same
    logits -- exact ties (duplicated bank rows, inside a level and across levels) included."""
    from hgrnet_b200 import ops
    h, x, train_index, n_levels, args, table, bank_train = _setup(levels, B, D, train_every)
    N = len(h)
    logits = _oracle_logits(x, bank_train, train_index, N)
    for target in sorted({N - 1, 0, N // 2, min(7, N - 1)}):
        L = len(h.c2p[target]) + 1
        counts = ops.new_hier_counts(DEV)
        lvl = torch.empty((B, n_levels), dtype=torch.int32, device=DEV)
        top1 = torch.empty((B,), dtype=torch.int32, device=DEV)
        ops.hier_metrics_fused_rows(x, targets=torch.full((B,), target, dtype=torch.int32, device=DEV), counts=counts,
                                    lvl_idx=lvl, top1=top1, **args, **table)
        want = torch.zeros_like(counts, device="cpu")
        want[L] = _oracle_bin(logits, train_index, h, target)
        assert torch.equal(counts.cpu(), want), (target, counts.cpu()[L], want[L])
        _check_winners(logits, train_index, h, lvl, top1)


def _mixed_targets(h, B, seed):
    """>= 5 labels, of 5 depths where the hierarchy has them (depth 0 included, so L = 1 occurs), spread over the
    rows; row 1 = -1 and row 3 = N are padding."""
    N = len(h)
    depths = sorted({0, 1, 2, h.max_depth // 2, h.max_depth - 1, h.max_depth} if h.max_depth >= 5 else range(h.max_depth + 1))
    g = torch.Generator().manual_seed(seed)
    labels = [h.d2n[d][int(torch.randint(len(h.d2n[d]), (1,), generator=g))] for d in depths] + [7, N - 1]
    t = torch.tensor([labels[i % len(labels)] for i in range(B)], dtype=torch.int32)
    t = t[torch.randperm(B, generator=g)]
    t[1], t[3] = -1, N
    return t


@pytest.mark.parametrize("levels,B,D,train_every", [((4, 20, 200), 64, 128, 1), ((3, 9, 40, 160), 33, 64, 2),
                                                    (_LEVELS20, 40, 64, 1), (_LEVELS12, 512, 1024, 1)])
def test_mixed_rows_match_oracle_per_label(levels, B, D, train_every):
    """A batch that mixes labels (padding rows included): bin L holds the oracle's counts of each label's sub-batch."""
    from hgrnet_b200 import ops
    h, x, train_index, n_levels, args, table, bank_train = _setup(levels, B, D, train_every)
    N = len(h)
    targets = _mixed_targets(h, B, seed=B)
    labels = sorted({int(t) for t in targets.tolist() if 0 <= t < N})
    assert len(labels) >= 5 and len({len(h.c2p[l]) for l in labels}) >= min(5, h.max_depth + 1)
    assert any(len(h.c2p[l]) == 0 for l in labels)

    # expected: the oracle on each label's sub-batch, in bin L; the padded rows nowhere
    logits = _oracle_logits(x, bank_train, train_index, N)
    want = torch.zeros((ops.HGR_HIER_MAX_CHAIN + 1, 4), dtype=torch.int64)
    for lab in labels:
        rows = (targets == lab).nonzero().flatten()
        want[len(h.c2p[lab]) + 1] += _oracle_bin(logits[rows], train_index, h, lab)

    t_dev = targets.to(DEV)
    got = ops.new_hier_counts(DEV)
    lvl = torch.empty((B, n_levels), dtype=torch.int32, device=DEV)
    top1 = torch.empty((B,), dtype=torch.int32, device=DEV)
    ops.hier_metrics_fused_rows(x, targets=t_dev, counts=got, lvl_idx=lvl, top1=top1, **args, **table)
    assert torch.equal(got.cpu(), want), (got.cpu()[got.cpu().any(1)], want[want.any(1)])
    assert int(want[:, 0].sum()) == B - 2

    # per-level winners and top-1 do not depend on the labels: those of every row, padding included, are the oracle's
    _check_winners(logits, train_index, h, lvl, top1)

    # the workspace came back zeroed: the same call again gives the same counters
    again = ops.new_hier_counts(DEV)
    ops.hier_metrics_fused_rows(x, targets=t_dev, counts=again, **args, **table)
    assert torch.equal(again, got)


def _opts(tmp_path, **kw):
    from hgrnet_b200.flags import parse_args
    o = parse_args([])
    o.device = 0
    o.folder = str(tmp_path / "out")
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _model(spec, tmp_path):
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import Hierarchy
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens
    h = Hierarchy(cases.tree_edges(spec["levels"], spec["tree_seed"]))
    n_nodes = len(h)
    test_ids = cases.test_ids(spec, n_nodes)
    enc = TableEncoder(cases.text_table(spec, n_nodes)).to(DEV)
    m = tree_model(_opts(tmp_path, weights="equal"), h.nodes, [h.nodes[i] for i in test_ids], clip_model=enc,
                   hierarchy=h, node_tokens=node_id_tokens(n_nodes)).to(DEV)
    m.update_classifier()
    return m, h, test_ids


@pytest.mark.parametrize("spec", cases.EVAL_CASES, ids=[s["name"] for s in cases.EVAL_CASES])
def test_update_rows_matches_oracle(spec, tmp_path):
    """``HierMetrics.update_rows`` over single-label batches against the sum of the oracle's per-batch increments."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import HierMetrics, _format
    model, h, test_ids = _model(spec, tmp_path)
    N = len(h)
    train_index = model.train_index.cpu()
    hm = HierMetrics(model)
    hits = ops.new_hits(DEV)
    n = 0
    tor = path = point = 0.0
    for feats, label in cases.eval_batches(spec, test_ids):
        x = model.encode_image_normalized(feats.to(DEV))
        tg = torch.full((feats.shape[0],), label, dtype=torch.long, device=DEV)
        model.score_topk(None, tg, hits=hits, feats_normalized=x)
        hm.update_rows(x, tg)
        a, b, c = orc.tor_por(_oracle_logits(x, model.bank_train, train_index, N), train_index, h.c2p, h.d2n, N, label)
        tor, path, point = tor + a, path + b, point + c
        n += feats.shape[0]
    want = (tor / n * 100.0, path / n * 100.0, point / n * 100.0)
    assert hm.path_all_count == n
    for a, b in zip(hm.ratios(n), want):
        assert abs(a - b) < 1e-9, (hm.ratios(n), want)
    assert _format(hits, n, hm) == _format(hits, n, types.SimpleNamespace(ratios=lambda _: want))


def test_eval_stream_hier_matches_eager(tmp_path):
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import HierMetrics
    spec = cases.EVAL_CASES[1]                                  # 6 levels, every node a test class, B = 37
    model, h, test_ids = _model(spec, tmp_path)
    N, B, slots = len(h), spec["B"], 4
    es = model.make_eval_stream(batch=B, slots=slots, streams=3, hier_metrics=True)
    g = torch.Generator().manual_seed(5)
    feats = [_emb(B, spec["D"], 300 + s, normalize=False) for s in range(slots)]
    labels = [torch.randint(0, N, (B,), generator=g, dtype=torch.int32) for _ in range(slots)]
    labels[2][0] = -1                                           # a padded row: scored by neither metric
    for s in range(slots):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for rep in range(3):
        for s in range(slots):
            es.step(s)
    es.end()

    hits = ops.new_hits(DEV)
    hm = HierMetrics(model)
    for rep in range(3):
        for s in range(slots):
            x = ops.normalize_rows(feats[s].to(DEV))
            t = labels[s].to(DEV)
            ops.score_topk(x, model.bank_test, col_id=model._test_index_i32, targets=t, K=20, hits=hits)
            hm.update_rows(x, t)
    assert es.hit_counts() == hits.tolist()
    assert es.host_hits.tolist() == hits.tolist()
    rows = 3 * (slots * B - 1)
    assert hm.path_all_count == rows
    got, want = es.hier_ratios(), hm.ratios(rows)
    assert all(abs(a - b) < 1e-9 for a, b in zip(got, want)), (got, want)
    assert want[0] > 0 and want[1] > 0 and want[2] > 0


def test_hier_rows_rejects_bad_arguments_and_counter_sets():
    from hgrnet_b200 import _cabi, ops
    from hgrnet_b200._cabi import HgrError
    h, x, train_index, n_levels, args, table, _ = _setup((4, 20, 200), 64, 128, 1)
    t = _mixed_targets(h, 64, seed=1).to(DEV)
    counts = ops.new_hier_counts(DEV)
    lib = _cabi.load()
    ends = (ctypes.c_int32 * n_levels)(*args["level_end"])
    ws = torch.zeros(64 * n_levels * 8 + 16, dtype=torch.uint8, device=DEV)
    p = lambda a: a.data_ptr()

    def call(chain_ptr=p(table["chain_ptr"]), n_lv=n_levels, level_end=ends, workspace=p(ws)):
        return lib.hgr_hier_metrics_fused_rows(p(x), p(args["bank_sorted"]), 64, args["bank_sorted"].shape[0], 128,
                                               level_end, n_lv, p(args["sorted_to_pos"]), p(args["first_out"]), p(t),
                                               len(h), chain_ptr, p(table["chain_pos"]), p(table["chain_level"]),
                                               None, 1, workspace, 64 * n_levels * 8, None, None, p(counts), None)

    for bad in (dict(chain_ptr=None), dict(workspace=p(ws) + 4)):
        with pytest.raises(HgrError):
            _cabi.check(call(**bad))
    M = args["bank_sorted"].shape[0]
    ends33 = (ctypes.c_int32 * 33)(*([0] * 32 + [M]))
    with pytest.raises(HgrError, match="levels"):
        _cabi.check(call(n_lv=33, level_end=ends33))
    args33 = dict(args, level_end=[0] * 32 + [M], first_out=torch.zeros(33, dtype=torch.int32, device=DEV))
    with pytest.raises(HgrError, match="levels"):                 # the same through ops
        ops.hier_metrics_fused_rows(x, targets=t, counts=counts, **args33, **table)
    assert counts.sum().item() == 0                              # nothing ran
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="need node_splits"):     # several counter sets, one per split
        ops.hier_metrics_fused_rows(x, targets=t, counts=ops.new_hier_counts(DEV, 2), **args, **table)
    cpu = {k: v.cpu() for k, v in table.items()}
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(x, targets=t, counts=counts, **args, **cpu)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(x.cpu(), targets=t, counts=counts, **args, **table)
