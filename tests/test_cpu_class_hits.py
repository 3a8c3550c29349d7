"""Per-class Hit@k (``hgr_class_hits`` / ``evaluate.ClassHits``), host side: a numpy oracle of the per-class table, the
arithmetic of ``class_summary`` / ``class_line``, the readout of ``EvalCounters`` on hand-built tables, the CLI flag
and the C ABI's argument checks.  The kernel is compared with this oracle in tests/test_gpu_class_hits.py."""
from __future__ import annotations

import numpy as np
import pytest
import torch

HIT_CUTS = (1, 2, 5, 10, 20)
COLS = len(HIT_CUTS) + 1


def oracle_class_counts(idx, targets, n_nodes, node_splits=None):
    """int64 ``[S, n_nodes, 6]`` table of ``idx`` ([B, K] or [S, B, K] node ids) against ``targets`` [B]: a row with a
    label in ``[0, n_nodes)`` adds 1 to ``rows`` of its label, and 1 to every Hit@k whose cut lies past the label's first
    position in the row's list (set s only when bit s of ``node_splits[label]`` is set)."""
    idx = np.asarray(idx)
    if idx.ndim == 2:
        idx = idx[None]
    S, B, K = idx.shape
    out = np.zeros((S, n_nodes, COLS), dtype=np.int64)
    for r in range(B):
        t = int(targets[r])
        if not 0 <= t < n_nodes:
            continue
        bits = 1 if node_splits is None else int(node_splits[t])
        for s in range(S):
            if not (bits >> s) & 1:
                continue
            out[s, t, -1] += 1
            where = np.nonzero(idx[s, r] == t)[0]
            if where.size:
                for i, k in enumerate(HIT_CUTS):
                    out[s, t, i] += int(where[0] < k)
    return out


def test_oracle_known_answers():
    # K = 6, 4 nodes: label 2 at position 0, at positions 3 and 4 (the first counts), absent; label 1 at position 5;
    # then the padding labels -1 and n_nodes
    idx = [[2, 0, 1, 3, -1, -1], [0, 1, 3, 2, 2, -1], [0, 1, 3, -1, -1, -1], [0, 3, 2, 3, 0, 1], [2, 2, 2, 2, 2, 2],
           [1, 1, 1, 1, 1, 1]]
    c = oracle_class_counts(idx, [2, 2, 2, 1, -1, 4], 4)[0]
    assert c[2].tolist() == [1, 1, 2, 2, 2, 3]
    assert c[1].tolist() == [0, 0, 0, 1, 1, 1]
    assert c[0].sum() == 0 and c[3].sum() == 0                       # -1 and 4 (= n_nodes) count nowhere
    # two sets, overlapping masks: node 2 in sets 0 and 1, node 1 in set 1 only
    two = oracle_class_counts(np.stack([idx, idx]), [2, 2, 2, 1, -1, 4], 4, node_splits=[0, 2, 3, 0])
    assert np.array_equal(two[0, 2], c[2]) and two[0, 1].sum() == 0
    assert np.array_equal(two[1], c)


def _table(rows):
    t = np.zeros((len(rows), COLS), dtype=np.int64)
    for i, r in enumerate(rows):
        t[i] = r
    return t


def test_class_summary_arithmetic():
    from hgrnet_b200.evaluate import class_line, class_summary
    # class 0: 10 rows, class 1: no rows (excluded), class 2: 2 rows, class 3: 5 rows
    t = _table([[5, 6, 8, 9, 10, 10], [0, 0, 0, 0, 0, 0], [0, 1, 1, 2, 2, 2], [1, 1, 2, 3, 5, 5]])
    s = class_summary(t)
    assert s["classes"] == 3
    want = [(5 / 10 + 0 / 2 + 1 / 5) / 3, (6 / 10 + 1 / 2 + 1 / 5) / 3, (8 / 10 + 1 / 2 + 2 / 5) / 3,
            (9 / 10 + 2 / 2 + 3 / 5) / 3, (10 / 10 + 2 / 2 + 5 / 5) / 3]
    assert [s["mean@%d" % k] for k in HIT_CUTS] == pytest.approx(want, rel=0, abs=1e-15)
    assert class_summary(torch.from_numpy(t)) == s                   # a tensor gives the same values
    assert class_line(s) == (" class_mean Top@1(%):23.33, Top@2(%):43.33, Top@5(%):56.67, Top@10(%):83.33, "
                             "Top@20(%):100.00 over 3 classes")
    # the image-weighted number of the same rows differs: 6 / 17 at top-1
    assert abs(t[:, 0].sum() / t[:, -1].sum() - s["mean@1"]) > 0.1
    z = class_summary(np.zeros((7, COLS), dtype=np.int64))
    assert z == {"classes": 0.0, **{"mean@%d" % k: 0.0 for k in HIT_CUTS}}
    assert class_line(z) == (" class_mean Top@1(%):0.00, Top@2(%):0.00, Top@5(%):0.00, Top@10(%):0.00, "
                             "Top@20(%):0.00 over 0 classes")
    with pytest.raises(ValueError):
        class_summary(np.zeros((3, 5), dtype=np.int64))
    with pytest.raises(ValueError):
        class_summary(np.zeros((2, 3, COLS), dtype=np.int64))


def test_eval_counters_readout_keeps_the_table_out_of_the_mirrored_buffer():
    from hgrnet_b200.evaluate import EvalCounters, class_line, class_summary, split_line
    n_nodes = 5
    plain = EvalCounters(torch.device("cpu"))
    one = EvalCounters(torch.device("cpu"), classes=n_nodes)
    assert one.counters.numel() == plain.counters.numel()            # the per-step copy keeps its size
    assert tuple(one.class_counts.shape) == (1, n_nodes, COLS)
    one.class_counts[0, 3] = torch.tensor([1, 2, 2, 2, 2, 4])
    assert one.class_table().tolist() == one.class_counts[0].tolist()
    assert one.class_summary() == class_summary(one.class_counts[0])
    with pytest.raises(RuntimeError):
        one.split_class_summary()
    with pytest.raises(RuntimeError):
        plain.class_table()
    three = EvalCounters(torch.device("cpu"), n_splits=3, classes=n_nodes)
    assert tuple(three.class_counts.shape) == (3, n_nodes, COLS)
    three.class_counts[1, 0] = torch.tensor([1, 1, 1, 1, 1, 1])
    three.split_counts[1] = torch.tensor([1, 1, 1, 1, 1, 1])
    lines = three.split_lines(["a", "b", "c"])
    assert lines[1] == split_line("b", [1] * 5, 1) + class_line(class_summary(three.class_counts[1]))
    assert lines[0].endswith("over 0 classes") and lines[1].endswith("over 1 classes")
    assert [s["classes"] for s in three.split_class_summary()] == [0, 1, 0]
    three.zero_()
    assert int(three.class_counts.abs().sum()) == 0 and int(three.counters.abs().sum()) == 0


def test_flag_parses_and_is_off_by_default():
    from hgrnet_b200.flags import parse_args
    assert parse_args([]).hgr_class_metrics is False
    assert parse_args(["--hgr_class_metrics", "True"]).hgr_class_metrics is True
    o = parse_args(["--hgr_class_metrics", "True", "--hgr_eval_splits", "hops2,hops3,rest"])
    assert o.hgr_class_metrics is True and o.hgr_eval_splits == "hops2,hops3,rest"


def test_ops_refuse_cpu_tensors():
    from hgrnet_b200 import ops
    with pytest.raises(ValueError, match="CUDA"):
        ops.class_hits(torch.zeros(4, 20, dtype=torch.int32), torch.zeros(4, dtype=torch.int32),
                       torch.zeros(1, 10, COLS, dtype=torch.int64))


def _abi(**kw):
    from hgrnet_b200 import _cabi
    a = dict(topk_idx=8, B=4, K=20, set_stride=80, n_sets=1, targets=8, node_splits=None, n_nodes=10, counts=8,
             stream=None)
    a.update(kw)
    return _cabi.load().hgr_class_hits(*a.values())


@pytest.mark.parametrize("bad", [dict(K=0), dict(K=33), dict(B=-1), dict(n_nodes=0), dict(n_nodes=1 << 31),
                                 dict(n_sets=2), dict(n_sets=9, node_splits=8), dict(n_sets=0),
                                 dict(n_sets=3, node_splits=8, set_stride=79), dict(topk_idx=None),
                                 dict(targets=None), dict(counts=None), dict(counts=12)])
def test_abi_rejects_bad_arguments(bad):
    assert _abi(**bad) == -1                                        # HGR_ERR_BAD_ARG, before any launch


def test_abi_zero_rows_is_a_no_op():
    assert _abi(B=0, topk_idx=None, targets=None, counts=None) == 0
