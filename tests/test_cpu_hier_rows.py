"""CPU tests of the host side of per-row TOR / POR (``hgr_hier_metrics_fused_rows``): the chain table that replaces
the per-batch Python chain, and the per-chain-length counters -> reference totals arithmetic."""
from __future__ import annotations

import ctypes
import os
import re
import time

import numpy as np
import pytest
import torch

from oracle import cases, hgr_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_table(h, train_ids):
    from hgrnet_b200.evaluate import chain_table
    ptr, pos, lvl = chain_table(h.c2p, h.depth, train_ids)
    assert ptr.dtype == pos.dtype == lvl.dtype == np.int32
    assert ptr.shape == (len(h) + 1,) and ptr[0] == 0 and ptr[-1] == pos.size == lvl.size
    pos_of = {int(n): j for j, n in enumerate(train_ids)}          # what HierMetrics.update builds per batch
    for n in range(len(h)):
        chain = list(h.c2p[n]) + [n]
        a, b = int(ptr[n]), int(ptr[n + 1])
        assert b - a == len(chain)
        assert pos[a:b].tolist() == [pos_of.get(p, -1) for p in chain], n
        assert lvl[a:b].tolist() == [len(h.c2p[p]) for p in chain], n


@pytest.mark.parametrize("name", ["quirky", "tree_4_20_200"])
def test_chain_table_matches_gen_tree(name, golden):
    from hgrnet_b200.hierarchy import Hierarchy
    edges = cases.QUIRKY_EDGES if name == "quirky" else cases.tree_edges([4, 20, 200], 3)
    h = Hierarchy(edges)
    assert h.c2p == golden["gen_tree"][name]["c2p"]                # the reference's chains, DAG included
    N = len(h)
    for train in (list(range(N)), list(range(0, N, 2)), [N - 1, 0, N - 1, 2]):   # all / every other / repeats, unsorted
        _check_table(h, train)


def test_chain_table_at_imagenet21k_scale():
    from hgrnet_b200.evaluate import chain_table
    from hgrnet_b200.hierarchy import WORDNET_LIKE_21841, synthetic_hierarchy
    h = synthetic_hierarchy(WORDNET_LIKE_21841, seed=1)
    leaves = h.d2n[h.max_depth][:1000]
    train = sorted(set(leaves) | {p for n in leaves for p in h.c2p[n]})   # 1,000 leaves + their ancestors
    t0 = time.perf_counter()
    chain_table(h.c2p, h.depth, train)
    assert time.perf_counter() - t0 < 0.5
    _check_table(h, train)
    _check_table(h, list(range(len(h))))


def test_hier_totals_hand_made():
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import hier_totals
    counts = torch.zeros((ops.HGR_HIER_MAX_CHAIN + 1, 4), dtype=torch.int64)
    counts[1] = torch.tensor([3, 2, 2, 2])       # L = 1: the single-node path counts its one match
    counts[3] = torch.tensor([2, 1, 5, 3])
    counts[32] = torch.tensor([1, 0, 31, 30])
    rows, hits, point, path = hier_totals(counts).tolist()
    assert (rows, hits) == (6, 3)
    assert point == pytest.approx(2 / 1 + 5 / 3 + 31 / 32, abs=1e-12)
    assert path == pytest.approx(2 / 1 + 3 / 2 + 30 / 31, abs=1e-12)
    assert hier_totals(torch.zeros_like(counts)).tolist() == [0.0, 0.0, 0.0, 0.0]


def test_hier_totals_reproduce_oracle_sums():
    """Single-label batches scored by oracle.tor_por (main.py:143,152-191), their integer counts put into bin L: the
    totals are the sums of the reference's per-batch path_add / point_add."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import hier_totals
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    h = synthetic_hierarchy([3, 9, 40, 160], seed=3)
    N = len(h)
    train_index = torch.arange(0, N, 2)
    counts = torch.zeros((ops.HGR_HIER_MAX_CHAIN + 1, 4), dtype=torch.int64)
    want_tor = want_path = want_point = 0.0
    rows = 0
    for b, target in enumerate([0, 1, 5, 20, 60, N - 1, N - 2, 2]):     # depths 0..3, two batches per length
        B = 7 + b
        g = torch.Generator().manual_seed(b)
        logits = torch.randn(B, N, generator=g).clamp_(-0.99, 0.99)
        logits[:, target] += 0.5 * torch.rand(B, generator=g)          # some rows hit their label
        tor, path_add, point_add = orc.tor_por(logits, train_index, h.c2p, h.d2n, N, target)
        L = len(h.c2p[target]) + 1
        edges = round(path_add * max(L - 1, 1))
        points = round(point_add * L)
        counts[L] += torch.tensor([B, int(tor), points, edges])
        want_tor, want_path, want_point, rows = want_tor + tor, want_path + path_add, want_point + point_add, rows + B
    assert (counts[1:5, 0] > 0).all()
    r, hits, point, path = hier_totals(counts).tolist()
    assert r == rows and hits == want_tor
    assert abs(path - want_path) < 1e-9 and abs(point - want_point) < 1e-9


def test_hier_max_chain_matches_header():
    from hgrnet_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "hgr_b200.h")).read()
    assert int(re.search(r"#define HGR_HIER_MAX_CHAIN (\d+)", header).group(1)) == _cabi.HGR_HIER_MAX_CHAIN == 32


@pytest.mark.parametrize("node_splits, n_sets", [(None, 0), (None, 2), (0x60000, 0), (0x60000, 9)])
def test_hier_rows_rejects_bad_counter_sets(node_splits, n_sets):
    """One counter set without node_splits, 1..8 with them: refused before any CUDA call (fake device pointers)."""
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    p = 0x10000
    ends = (ctypes.c_int32 * 2)(10, 40)
    assert lib.hgr_hier_metrics_fused_rows(p, p, 64, 40, 128, ends, 2, p, p, p, 600, p, p, p, node_splits, n_sets, p,
                                           64 * 2 * 8, None, None, p, None) == -1
    assert "counter sets" in lib.hgr_last_error().decode()


def test_new_hier_counts_shapes():
    from hgrnet_b200 import ops
    assert tuple(ops.new_hier_counts("cpu").shape) == (ops.HGR_HIER_MAX_CHAIN + 1, 4)
    assert tuple(ops.new_hier_counts("cpu", 3).shape) == (3, ops.HGR_HIER_MAX_CHAIN + 1, 4)


def test_hier_rows_refuses_cpu_tensors():
    from hgrnet_b200 import ops
    z = lambda *s, dt=torch.int32: torch.zeros(*s, dtype=dt)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(z(4, 64, dt=torch.bfloat16), z(8, 64, dt=torch.bfloat16), [8], z(8), z(1), z(4),
                                    z(9), z(8), z(8), ops.new_hier_counts("cpu"))


def test_eval_counters_layout_and_readout():
    """``EvalCounters``: hits, then per-split hits, then TOR / POR sets, then mistake sets in one int64 buffer (the
    byte layout the streams mirror to the host), and the ratios / lines derived from it."""
    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import EvalCounters, hier_line, split_line
    H, NH, MC = (ops.HGR_HIER_MAX_CHAIN + 1) * 4, ops.HGR_NUM_HITS, ops.HGR_MISTAKE_COUNTERS
    one = EvalCounters("cpu", hier=True, mistakes=True)
    assert one.counters.numel() == NH + H + MC and one.split_counts is None
    assert one.hier_counts.shape == (1, ops.HGR_HIER_MAX_CHAIN + 1, 4) and one.mistake_counts.shape == (1, MC)
    assert one.hier_counts.data_ptr() == one.counters[NH:].data_ptr()
    one.hier_counts[0, 3] = torch.tensor([4, 2, 6, 4])             # 4 rows with 3-entry chains
    assert one.hier_ratios() == (50.0, 50.0, 50.0)
    assert EvalCounters("cpu", hier=True).hier_ratios() == (0.0, 0.0, 0.0)
    with pytest.raises(RuntimeError):
        one.split_hit_counts()
    S = 3
    read = []
    c = EvalCounters("cpu", n_splits=S, hier=True, read=lambda x: read.append(1) or 2 * x)
    assert c.counters.numel() == NH + S * (NH + 1) + S * H and c.mistake_counts is None
    assert c.split_counts.data_ptr() == c.counters[NH:].data_ptr()
    assert c.hier_counts.data_ptr() == c.counters[NH + S * (NH + 1):].data_ptr()
    c.split_counts[1] = torch.tensor([1, 2, 3, 4, 5, 10])
    c.hier_counts[1, 1] = torch.tensor([5, 1, 2, 3])               # single-node chains: path = edges
    assert c.split_hit_counts()[1] == [2, 4, 6, 8, 10, 20]         # through the read step
    assert c.split_ratios()[1] == (20.0, 60.0, 40.0) and c.split_ratios()[0] == (0.0, 0.0, 0.0)
    lines = c.split_lines(["a", "b", "c"])
    assert lines[1] == split_line("b", [2, 4, 6, 8, 10], 20, (2.0, 4.0, 6.0, 10.0))
    assert lines[1].endswith(hier_line(10.0, 60.0, 20.0)) and lines[0].startswith("a: Top@1(%):0.00")
    with pytest.raises(RuntimeError):
        c.hier_ratios()
    with pytest.raises(RuntimeError):
        c.split_mistake_summary()
    assert len(read) == 4                                           # one read step per readout
