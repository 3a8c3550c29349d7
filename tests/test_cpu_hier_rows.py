"""CPU tests of the host side of per-row TOR / POR (``hgr_hier_metrics_fused_rows``): the chain table that replaces
the per-batch Python chain, and the per-chain-length counters -> reference totals arithmetic."""
from __future__ import annotations

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


def test_hier_rows_refuses_cpu_tensors():
    from hgrnet_b200 import ops
    z = lambda *s, dt=torch.int32: torch.zeros(*s, dtype=dt)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.hier_metrics_fused_rows(z(4, 64, dt=torch.bfloat16), z(8, 64, dt=torch.bfloat16), [8], z(8), z(1), z(4),
                                    z(9), z(8), z(8), ops.new_hier_counts("cpu"))
