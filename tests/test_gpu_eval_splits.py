"""Several test splits in one scoring pass (``hgr_score_topk_splits`` / ``hgr_hier_metrics_fused_rows`` with ``node_splits`` /
``evaluate.SplitEval``): per split the same top-K, hits and row counts as ``score_topk`` on that split's rows of the
union bank, the fp32 oracle under the tie-aware comparison, exact repairs on a hierarchy-ordered bank, per-split TOR /
POR counters, and the multi-split CLI path."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import compare_topk, hostile_bank

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _unit(n, d, seed):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    return (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)


def _splits(kind, n_nodes, C, seed=0):
    """Node ids of the test classes (a random C-subset of the nodes) and splits over them: 'hops' = three nested sets of
    C * 1549/20842, C * 7860/20842 and C classes; 'overlap' = three overlapping sets that are not nested."""
    g = np.random.default_rng(seed)
    nodes = g.choice(n_nodes, size=C, replace=False)
    if kind == "hops":
        a, b = max(1, C * 1549 // 20842), max(2, C * 7860 // 20842)
        return {"2-hops": nodes[:a], "3-hops": nodes[:b], "all": nodes}
    third = C // 3
    return {"a": nodes[:2 * third], "b": nodes[third:], "c": np.concatenate([nodes[:third // 2], nodes[-third // 2:]])}


def _layout(splits, n_nodes, bank_rows):
    from hgrnet_b200.evaluate import split_groups
    names, bank_nodes, ends, masks, node_splits = split_groups(splits, n_nodes)
    bank = bank_rows[torch.from_numpy(bank_nodes)].to(DEV).contiguous()
    return names, bank_nodes, ends, masks, node_splits, bank


def _run(kind, B, D, n_nodes, C, bank_kind="iid", x=None):
    from hgrnet_b200 import ops
    splits = _splits(kind, n_nodes, C)
    all_rows = hostile_bank(n_nodes, D, bank_kind) if bank_kind != "iid" else _unit(n_nodes, D, 5)
    names, bank_nodes, ends, masks, node_splits, bank = _layout(splits, n_nodes, all_rows)
    if bank_kind != "iid":   # hierarchy order: keep the rows of every group in node order (no permutation)
        order = np.concatenate([np.sort(bank_nodes[b:e]) for b, e in zip([0] + ends[:-1], ends)])
        bank_nodes = order
        bank = all_rows[torch.from_numpy(order)].to(DEV).contiguous()
    col_id = torch.from_numpy(bank_nodes).to(torch.int32).to(DEV)
    union = bank_nodes
    g = torch.Generator().manual_seed(7)
    targets = torch.from_numpy(union[torch.randint(0, len(union), (B,), generator=g).numpy()]).to(torch.int32).to(DEV)
    if x is None:
        x = ops.normalize_rows((bank[torch.randint(0, len(union), (B,), generator=g).to(DEV)].float()
                                + 0.5 * torch.randn(B, D, generator=g).to(DEV) / D ** 0.5))
    S = len(names)
    counts = torch.zeros((S, ops.HGR_NUM_HITS + 1), dtype=torch.int64, device=DEV)
    ns = torch.from_numpy(node_splits).to(DEV)
    val, idx = ops.score_topk_splits(x, bank, ends, masks, S, col_id=col_id, targets=targets, node_splits=ns,
                                     counts=counts)
    rescans = ops.last_rescan_count()
    return dict(x=x, bank=bank, col_id=col_id, targets=targets, ends=ends, masks=masks, node_splits=node_splits,
                val=val, idx=idx, counts=counts.cpu(), rescans=rescans, S=S)


def _split_rows(r, s):
    """Bank rows of split s in union order (the concatenation of its groups)."""
    ends, masks = r["ends"], r["masks"]
    rows = [torch.arange(b, e) for b, e, m in zip([0] + ends[:-1], ends, masks) if (m >> s) & 1]
    return torch.cat(rows).to(DEV)


def _check_against_single(r, need_bitwise):
    from hgrnet_b200 import ops
    x, targets = r["x"], r["targets"]
    in_s_all = torch.from_numpy(r["node_splits"]).to(DEV)[targets.long()]
    for s in range(r["S"]):
        rows = _split_rows(r, s)
        sub, sub_id = r["bank"][rows].contiguous(), r["col_id"][rows].contiguous()
        in_s = ((in_s_all >> s) & 1).bool()
        t = torch.where(in_s, targets, torch.full_like(targets, -1))
        hits = ops.new_hits(DEV)
        v1, i1 = ops.score_topk(x, sub, col_id=sub_id, targets=t, hits=hits)
        single_rescans = ops.last_rescan_count()
        if need_bitwise and single_rescans == 0 and r["rescans"] == 0:
            assert torch.equal(i1, r["idx"][s]), "split %d: ids differ from score_topk on the split's rows" % s
            assert torch.equal(v1, r["val"][s]), "split %d: values differ from score_topk on the split's rows" % s
        assert r["counts"][s, :ops.HGR_NUM_HITS].tolist() == hits.tolist(), "split %d hits" % s
        assert int(r["counts"][s, ops.HGR_NUM_HITS]) == int(in_s.sum()), "split %d rows" % s
        logits = (x.float() @ sub.float().T).cpu()
        compare_topk(r["val"][s], r["idx"][s], logits, sub_id.cpu(), 20)


@pytest.mark.parametrize("kind", ["hops", "overlap"])
@pytest.mark.parametrize("B,D,n_nodes,C", [(256, 512, 4000, 2900), (512, 1024, 21841, 20842)])
def test_splits_equal_per_split_runs(kind, B, D, n_nodes, C):
    r = _run(kind, B, D, n_nodes, C)
    assert r["rescans"] == 0
    _check_against_single(r, need_bitwise=True)


def test_hostile_bank_is_repaired_exactly():
    # overlapping splits of 1/3 - 2/3 of the classes get narrow lists; rows of a group in hierarchy order defeat them
    r = _run("overlap", 512, 512, 22000, 20842, bank_kind="clustered")
    assert r["rescans"] > 0, "a hierarchy-ordered bank should need exact repairs"
    _check_against_single(r, need_bitwise=False)


def test_one_split_equals_score_topk():
    from hgrnet_b200 import ops
    x = _unit(384, 512, 1).to(DEV)
    bank = _unit(5000, 512, 2).to(DEV)
    v, i = ops.score_topk_splits(x, bank, [5000], [1], 1, id_base=3)
    v1, i1 = ops.score_topk(x, bank, id_base=3)
    assert torch.equal(i[0], i1) and torch.equal(v[0], v1)


def test_tor_por_split_sets_match_single_set_calls():
    from hgrnet_b200 import ops
    from tests.test_gpu_hier_rows import _setup
    h, x, train_index, n_levels, args, table, _ = _setup((4, 20, 160, 900), 300, 256, 2)
    N = len(h)
    g = torch.Generator().manual_seed(4)
    targets = torch.randint(-1, N, (x.shape[0],), generator=g).to(torch.int32).to(DEV)
    node_splits = torch.randint(0, 8, (N,), generator=g).to(torch.uint8).to(DEV)   # three splits, any overlap
    counts = ops.new_hier_counts(DEV, 3)
    ops.hier_metrics_fused_rows(x, targets=targets, node_splits=node_splits, counts=counts, **args, **table)
    for s in range(3):
        in_s = (targets >= 0) & ((node_splits[targets.clamp(min=0).long()] >> s) & 1).bool()
        ref = ops.new_hier_counts(DEV)
        ops.hier_metrics_fused_rows(x[in_s].contiguous(), targets=targets[in_s].contiguous(), counts=ref, **args,
                                    **table)
        assert torch.equal(counts[s], ref), "split %d" % s


def test_main_cli_with_eval_splits(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "main.py"), "--train", "False", "--hgr_synthetic", "10,100,1000",
           "--hgr_eval_splits", "hops2,hops3,rest", "--folder", str(tmp_path), "--test_batch_size", "256",
           "--weights", str(tmp_path / "w")]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for name in ("hops2", "hops3", "rest"):
        assert ("\n%s: Top@1(%%)" % name) in out.stdout, out.stdout[-2000:]


@pytest.mark.parametrize("bank_kind", ["iid", "dups"])
def test_tiny_groups_and_ties(bank_kind):
    """Groups of one row and of fewer than K rows, next to a large one; with 'dups' every bank row has 39 exact copies,
    so ties straddle the group boundaries and the (value desc, bank row asc) order decides."""
    from hgrnet_b200 import ops
    n_nodes, D, B = 3000, 256, 300
    nodes = np.random.default_rng(3).choice(n_nodes, size=2500, replace=False)
    splits = {"one": nodes[:1], "few": nodes[:7], "all": nodes, "odd": nodes[1:23]}
    rows = hostile_bank(n_nodes, D, bank_kind) if bank_kind != "iid" else _unit(n_nodes, D, 9)
    names, bank_nodes, ends, masks, node_splits, bank = _layout(splits, n_nodes, rows)
    assert min(e - b for b, e in zip([0] + ends[:-1], ends)) == 1
    col_id = torch.from_numpy(bank_nodes).to(torch.int32).to(DEV)
    g = torch.Generator().manual_seed(8)
    targets = torch.from_numpy(bank_nodes[torch.randint(0, len(bank_nodes), (B,), generator=g).numpy()])
    targets[:40] = int(nodes[0])                                         # rows of the one-class split
    targets = targets.to(torch.int32).to(DEV)
    x = ops.normalize_rows(bank[torch.randint(0, len(bank_nodes), (B,), generator=g).to(DEV)].float()
                           + 0.3 * torch.randn(B, D, generator=g).to(DEV) / D ** 0.5)
    counts = torch.zeros((len(names), ops.HGR_NUM_HITS + 1), dtype=torch.int64, device=DEV)
    val, idx = ops.score_topk_splits(x, bank, ends, masks, len(names), col_id=col_id, targets=targets,
                                     node_splits=torch.from_numpy(node_splits).to(DEV), counts=counts)
    r = dict(x=x, bank=bank, col_id=col_id, targets=targets, ends=ends, masks=masks, node_splits=node_splits, val=val,
             idx=idx, counts=counts.cpu(), rescans=ops.last_rescan_count(), S=len(names))
    _check_against_single(r, need_bitwise=True)
    assert int(r["counts"][0, 0]) == 40 and int(r["counts"][0, ops.HGR_NUM_HITS]) == 40   # one class: always Top@1


def _stream_model(tmp_path):
    from oracle import cases
    from tests.test_gpu_hier_rows import _model
    spec = cases.EVAL_CASES[1]                                  # 6 levels, every node a test class, B = 37
    model, h, test_ids = _model(spec, tmp_path)
    return spec, model, h


def test_eval_stream_splits_match_eager_counter_block(tmp_path):
    """A captured ``EvalStream(splits=...)``, replayed over several slots and streams, gives the counters of the eager
    ``SplitEval.update`` calls: per split hits / rows and TOR / POR."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import SplitEval, hier_totals
    spec, model, h = _stream_model(tmp_path)
    N, B, slots = len(h), spec["B"], 4
    ids = np.random.default_rng(1).permutation(N)
    splits = {"small": ids[:30], "half": ids[:N // 2], "other": ids[N // 3:]}
    es = model.make_eval_stream(batch=B, slots=slots, streams=3, hier_metrics=True, eval_splits=splits)
    g = torch.Generator().manual_seed(6)
    feats = [torch.randn(B, spec["D"], generator=g) for _ in range(slots)]
    labels = [torch.from_numpy(ids[torch.randint(0, N, (B,), generator=g).numpy()]).to(torch.int32)
              for _ in range(slots)]
    labels[1][:10] = torch.from_numpy(ids[:10]).to(torch.int32)  # rows of the small split
    labels[2][0] = -1                                           # a padded row: counted nowhere
    for s in range(slots):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for rep in range(3):
        for s in range(slots):
            es.step(s)
    es.end()

    se = SplitEval(model, splits, hier=True)
    for rep in range(3):
        for s in range(slots):
            se.update(ops.normalize_rows(feats[s].to(DEV)), labels[s].to(DEV))
    want = se.hit_counts()
    assert es.split_hit_counts() == want
    assert es.host_counters[ops.HGR_NUM_HITS:].tolist() == es.counters[ops.HGR_NUM_HITS:].tolist()
    assert all(w[ops.HGR_NUM_HITS] > 0 for w in want)
    assert torch.equal(es.hier_counts, se.hier_counts)
    acc = hier_totals(se.hier_counts).tolist()
    for (hr, pr, por), (rows, tor, point, path) in zip(es.split_ratios(), acc):
        assert rows > 0
        assert abs(hr - tor / rows * 100.0) < 1e-9 and abs(pr - path / rows * 100.0) < 1e-9
        assert abs(por - point / rows * 100.0) < 1e-9


def test_evaluate_test_lines_match_oracle_per_split(tmp_path, monkeypatch):
    """``evaluate.test`` with ``--hgr_eval_splits``: the line of each split is the line the oracle's restatement of the
    reference's ``main.test`` prints for that split alone -- model_test = the split's classes, only the batches whose
    label is in the split, TOR / POR against the batch's label (main.py:104-222)."""
    import re
    from hgrnet_b200 import evaluate
    from hgrnet_b200.synthetic import FeatureLoader
    from oracle import cases, hgr_oracle as orc
    monkeypatch.chdir(tmp_path)
    spec = dict(cases.EVAL_CASES[1], batches=10)
    model, h, test_ids = __import__("tests.test_gpu_hier_rows", fromlist=["_model"])._model(spec, tmp_path)
    N = len(h)
    batches = cases.eval_batches(spec, test_ids)
    labels = [l for _, l in batches]
    rng = np.random.default_rng(2)
    extra = rng.permutation(N)
    split_ids = {"s0": sorted(set(labels[:3]) | set(extra[:20].tolist())),
                 "s1": sorted(set(labels[2:7]) | set(extra[20:90].tolist())),
                 "all": list(range(N))}
    opts = model.opts
    opts.print_freq = 1000
    opts.hgr_eval_splits = "s0,s1,all"
    out = evaluate.test(opts, model, DEV, splits={k: [h.nodes[i] for i in v] for k, v in split_ids.items()},
                        loader=FeatureLoader([f for f, _ in batches], labels))
    lines = {l.split(": ", 1)[0]: l.split(": ", 1)[1] for l in out.strip().split("\n")}
    assert list(lines) == ["s0", "s1", "all"]
    obank = orc.normalize_rows(cases.text_table(spec, N))
    train_index = torch.arange(N)
    for name, ids in split_ids.items():
        test_index = torch.tensor(ids)
        hits = {k: 0 for k in orc.TOPK}
        tor = path = point = 0.0
        n = ties = 0
        for feats, label in batches:
            if label not in set(ids):
                continue
            lg = orc.forward_logits(feats, obank)
            _, vals, hh = orc.eval_hits(lg, test_index, torch.full((feats.shape[0],), label))
            for k in hits:
                hits[k] += hh[k]
            a, b, c = orc.tor_por(lg, train_index, h.c2p, h.d2n, N, label)
            tor, path, point = tor + a, path + b, point + c
            n += feats.shape[0]
            top = lg[:, test_index].topk(min(21, len(ids)), 1, True, True)[0]
            ties += int(((top[:, :-1] - top[:, 1:]) <= 2e-3).any(1).sum())
        s, _ = orc.count_acc(hits, n)
        want = s + " hit_ratio(%):{:.2f}".format(tor / n * 100.0) + " path_ratio(%):{:.2f}".format(path / n * 100.0) \
            + " point_ratio(%):{:.2f}".format(point / n * 100.0)
        got = lines[name]
        if ties == 0:
            assert got[: got.index(" hit_ratio")] == want[: want.index(" hit_ratio")], (name, got, want)
        mine = [float(v) for v in re.findall(r":(-?\d+\.\d+)", got)]
        ref = [float(v) for v in re.findall(r":(-?\d+\.\d+)", want)]
        slack = 100.0 * (ties + 2) / n
        assert len(mine) == len(ref) == 8
        assert all(abs(a - b) <= slack + 0.011 for a, b in zip(mine, ref)), (name, got, want)
