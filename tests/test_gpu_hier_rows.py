"""TOR / POR with one label per row (``hgr_hier_metrics_fused_rows``, main.py:143,152-191): against the single-label
fused call on each label's sub-batch, against ``HierMetrics.update_fused`` on single-label batches, and inside the
graph-replayed ``EvalStream``."""
from __future__ import annotations

import ctypes

import pytest
import torch

from oracle import cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _emb(n, d, seed, normalize=True):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    if normalize:
        x = x / x.norm(dim=-1, keepdim=True)
    return x.to(torch.bfloat16).float()


def _setup(levels, B, D, train_every):
    """The inputs of test_hier_metrics_fused_matches_dense_pass (tests/test_gpu_kernels.py), duplicated bank rows
    included, plus the chain table."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import chain_table
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    h = synthetic_hierarchy(list(levels), seed=3)
    N = len(h)
    bank = _emb(N, D, 21).to(torch.bfloat16)
    bank[5] = bank[3]
    bank[N - 2] = bank[N // 2]
    bank[7] = bank[N - 1]                                       # a tie across two levels
    x = ops.normalize_rows(_emb(B, D, 22, normalize=False).to(DEV))
    train_index = torch.arange(0, N, train_every)
    depth = torch.from_numpy(h.depth).long()
    n_levels = int(depth.max()) + 1
    dt = depth[train_index]
    M = len(train_index)
    first_out = torch.tensor([int((dt != l).nonzero()[0]) if (dt != l).any() else M for l in range(n_levels)],
                             dtype=torch.int32, device=DEV)
    order = torch.sort(dt, stable=True).indices
    args = dict(bank_sorted=bank[train_index].to(DEV)[order.to(DEV)].contiguous(),
                level_end=torch.cumsum(torch.bincount(dt, minlength=n_levels), 0).tolist(),
                sorted_to_pos=order.to(torch.int32).to(DEV), first_out=first_out)
    table = [torch.from_numpy(a).to(DEV) for a in chain_table(h.c2p, h.depth, train_index.tolist())]
    return h, x, train_index, n_levels, args, dict(zip(("chain_ptr", "chain_pos", "chain_level"), table))


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
                                                    (tuple(1 + i // 2 for i in range(20)), 40, 64, 1),
                                                    ((20, 150, 900, 3000, 5500, 5500, 3500, 1800, 900, 400, 120, 51), 512, 1024, 1)])
def test_rows_equal_per_label_calls(levels, B, D, train_every):
    from hgrnet_b200 import ops
    h, x, train_index, n_levels, args, table = _setup(levels, B, D, train_every)
    N = len(h)
    targets = _mixed_targets(h, B, seed=B)
    pos_of = {int(n): j for j, n in enumerate(train_index.tolist())}
    labels = sorted({int(t) for t in targets.tolist() if 0 <= t < N})
    assert len(labels) >= 5 and len({len(h.c2p[l]) for l in labels}) >= min(5, h.max_depth + 1)
    assert any(len(h.c2p[l]) == 0 for l in labels)

    # expected: ops.hier_metrics_fused on each label's sub-batch, in bin L; the padded rows nowhere
    want = torch.zeros((ops.HGR_HIER_MAX_CHAIN + 1, 4), dtype=torch.int64)
    for lab in labels:
        rows = (targets == lab).nonzero().flatten()
        parents = list(h.c2p[lab]) + [lab]
        c = torch.zeros(3, dtype=torch.int64, device=DEV)
        ops.hier_metrics_fused(x[rows.to(DEV)].contiguous(), args["bank_sorted"], args["level_end"], args["sorted_to_pos"],
                               args["first_out"], torch.tensor([pos_of.get(p, -1) for p in parents], dtype=torch.int32, device=DEV),
                               torch.tensor([len(h.c2p[p]) for p in parents], dtype=torch.int32, device=DEV), c)
        want[len(parents)] += torch.cat([torch.tensor([rows.numel()]), c.cpu()])

    t_dev = targets.to(DEV)
    got = ops.new_hier_counts(DEV)
    lvl = torch.empty((B, n_levels), dtype=torch.int32, device=DEV)
    top1 = torch.empty((B,), dtype=torch.int32, device=DEV)
    ops.hier_metrics_fused_rows(x, targets=t_dev, counts=got, lvl_idx=lvl, top1=top1, **args, **table)
    assert torch.equal(got.cpu(), want), (got.cpu()[got.cpu().any(1)], want[want.any(1)])
    assert int(want[:, 0].sum()) == B - 2

    # per-level winners and top-1 do not depend on the labels: a single-label call on the full batch
    lvl1 = torch.empty_like(lvl)
    top11 = torch.empty_like(top1)
    ops.hier_metrics_fused(x, args["bank_sorted"], args["level_end"], args["sorted_to_pos"], args["first_out"],
                           torch.tensor([0], dtype=torch.int32, device=DEV), torch.tensor([0], dtype=torch.int32, device=DEV),
                           torch.zeros(3, dtype=torch.int64, device=DEV), lvl_idx=lvl1, top1=top11)
    assert torch.equal(lvl, lvl1) and torch.equal(top1, top11)

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
def test_update_rows_reproduces_update_fused(spec, tmp_path):
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import HierMetrics, _format
    model, h, test_ids = _model(spec, tmp_path)
    hm_f, hm_r = HierMetrics(model), HierMetrics(model)
    hits = ops.new_hits(DEV)
    n = 0
    for feats, label in cases.eval_batches(spec, test_ids):
        x = model.encode_image_normalized(feats.to(DEV))
        tg = torch.full((feats.shape[0],), label, dtype=torch.long, device=DEV)
        model.score_topk(None, tg, hits=hits, feats_normalized=x)
        hm_f.update_fused(x, label)
        hm_r.update_rows(x, tg)
        n += feats.shape[0]
    assert hm_r.path_all_count == hm_f.path_all_count == n
    for a, b in zip(hm_r.ratios(n), hm_f.ratios(n)):
        assert abs(a - b) < 1e-9, (hm_r.ratios(n), hm_f.ratios(n))
    assert _format(hits, n, hm_r) == _format(hits, n, hm_f)


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


def test_hier_rows_rejects_bad_arguments():
    from hgrnet_b200 import _cabi, ops
    from hgrnet_b200._cabi import HgrError
    h, x, train_index, n_levels, args, table = _setup((4, 20, 200), 64, 128, 1)
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
                                               workspace, 64 * n_levels * 8, None, None, p(counts), None)

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
    cpu = {k: v.cpu() for k, v in table.items()}
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(x, targets=t, counts=counts, **args, **cpu)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(x.cpu(), targets=t, counts=counts, **args, **table)
