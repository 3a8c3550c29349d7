"""Host logic of the multi-split evaluation (``evaluate.split_groups`` / ``evaluate.split_line``): grouping of the union
by split membership, group order, the fixed permutation inside each group, the per-node split bits, and the per-split
line format against the oracle's ``count_acc``."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from hgrnet_b200.evaluate import split_groups, split_line
from oracle import hgr_oracle as orc


def test_groups_by_membership():
    splits = {"2-hops": [7, 3], "3-hops": [3, 7, 10, 12], "all": [3, 7, 10, 12, 1, 20]}
    names, bank_nodes, ends, masks, node_splits = split_groups(splits, 25)
    assert names == ["2-hops", "3-hops", "all"]
    assert masks == [0b100, 0b110, 0b111]                  # ascending membership mask
    assert ends == [2, 4, 6]
    groups = [set(bank_nodes[b:e].tolist()) for b, e in zip([0] + ends[:-1], ends)]
    assert groups == [{1, 20}, {10, 12}, {3, 7}]
    assert node_splits.dtype == np.uint8 and node_splits.shape == (25,)
    assert node_splits[3] == 0b111 and node_splits[10] == 0b110 and node_splits[20] == 0b100 and node_splits[0] == 0
    for s, name in enumerate(names):                         # the groups of split s hold exactly its classes
        rows = np.concatenate([bank_nodes[b:e] for b, e, m in zip([0] + ends[:-1], ends, masks) if (m >> s) & 1])
        assert sorted(rows.tolist()) == sorted(splits[name])


def test_permutation_inside_groups_is_fixed_and_not_identity():
    rng = np.random.default_rng(0)
    nodes = rng.choice(5000, size=3000, replace=False)
    splits = {"a": nodes[:2000], "b": nodes[1000:]}
    a = split_groups(splits, 5000)
    b = split_groups(splits, 5000)
    assert np.array_equal(a[1], b[1]) and a[2] == b[2]
    for lo, hi in zip([0] + a[2][:-1], a[2]):
        grp = a[1][lo:hi]
        assert not np.array_equal(grp, np.sort(grp))     # pseudo-random, not node order
    assert a[3] == [0b01, 0b10, 0b11]


def test_split_limits():
    with pytest.raises(ValueError):
        split_groups({str(i): [i] for i in range(9)}, 20)       # more than 8 splits
    with pytest.raises(ValueError):
        split_groups({"a": []}, 20)
    # 5 splits over single classes with 17 distinct memberships -> more than 16 groups
    splits = {str(s): [n for n in range(1, 18) if (n >> s) & 1] for s in range(5)}
    with pytest.raises(ValueError):
        split_groups(splits, 40)


def test_split_line_matches_count_acc():
    hits = [3, 5, 9, 12, 17]
    ref, _ = orc.count_acc(dict(zip((1, 2, 5, 10, 20), hits)), 40)
    assert split_line("3-hops", hits, 40) == "3-hops: " + ref
    line = split_line("all", hits, 40, (10.0, 20.0, 15.0, 38))
    assert line == "all: " + ref + " hit_ratio(%):25.00 path_ratio(%):39.47 point_ratio(%):50.00"
