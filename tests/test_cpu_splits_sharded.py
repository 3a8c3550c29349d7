"""CPU tests of several test splits on the class-sharded head (``dist.split_shard_bounds`` / ``dist.SplitShard`` /
``hgr_score_topk_splits_scatter_bounded``): the per-group cut of the union bank, the exchange-slot layout with split
areas, the per-split global list lengths and the argument checks that fire before any CUDA call."""
from __future__ import annotations

import pytest
import torch

# cfg 5 with the nested 2-hops / 3-hops / all splits of tools/bench_eval_splits.py: groups in ascending mask order
CFG5_ENDS, CFG5_MASKS, CFG5_SPLIT_C = [12982, 19293, 20842], [4, 6, 7], [1549, 7860, 20842]


@pytest.mark.parametrize("group_end,world", [([5], 1), ([5], 2), ([100, 130, 400], 3), (CFG5_ENDS, 8),
                                             (CFG5_ENDS, 16), ([3, 5, 12], 8), ([1, 2, 3, 4], 16), ([7], 8),
                                             ([1000], 3), ([2, 40, 41, 700], 2)])
def test_split_shard_bounds_partition_every_group(group_end, world):
    from hgrnet_b200.dist import split_shard_bounds
    parts = split_shard_bounds(group_end, world)
    assert len(parts) == world
    begins = [0] + group_end[:-1]
    seen = []
    per_group = [[0] * world for _ in group_end]
    for r, (ranges, local_end, kept) in enumerate(parts):
        assert len(ranges) == len(local_end) == len(kept)
        assert kept == sorted(set(kept))                                 # group order kept
        assert all(b < a for b, a in zip(local_end, local_end[1:]))      # strictly ascending: empties dropped
        n = 0
        for (lo, hi), e, g in zip(ranges, local_end, kept):
            assert begins[g] <= lo < hi <= group_end[g]                  # a slice of its own group
            n += hi - lo
            assert e == n
            per_group[g][r] = hi - lo
            seen += list(range(lo, hi))
    assert sorted(seen) == list(range(group_end[-1])) and len(seen) == len(set(seen))   # every row on exactly one rank
    for g, counts in enumerate(per_group):
        assert max(counts) - min(counts) <= 1                            # balanced to within one row per group
        assert sum(counts) == group_end[g] - begins[g]


def test_split_shard_bounds_small_groups_and_empty_ranks():
    from hgrnet_b200.dist import split_shard_bounds
    parts = split_shard_bounds([1, 2], 3)                                # two one-row groups over three ranks
    assert [p[1] for p in parts] == [[], [], [1, 2]]
    assert parts[0] == ([], [], [])                                      # a rank without rows
    parts = split_shard_bounds([3, 5], 4)                                # groups of 3 and 2 rows: some ranks miss one
    assert [p[2] for p in parts] == [[], [0, 1], [0], [0, 1]]
    assert [p[1] for p in parts] == [[], [1, 2], [1], [1, 2]]
    assert split_shard_bounds([9], 1) == [([(0, 9)], [9], [0])]          # one rank: the union bank itself


def test_cfg5_rows_per_rank():
    from hgrnet_b200.dist import split_shard_bounds
    for ranges, local_end, kept in split_shard_bounds(CFG5_ENDS, 8):
        sizes = [hi - lo for lo, hi in ranges]
        assert kept == [0, 1, 2]
        assert [abs(a - b) <= 1 for a, b in zip(sizes, (12982 / 8, 6311 / 8, 1549 / 8))] == [True] * 3


class _FakeSplitEval:
    """What ``SplitShard`` needs of an ``evaluate.SplitEval``."""

    def __init__(self, group_end, masks, n_nodes, D=16, hier=None):
        self.group_end, self.group_splits = group_end, masks
        self.S = max(m.bit_length() for m in masks)
        self.names = ["s%d" % s for s in range(self.S)]
        C = group_end[-1]
        self.col_id = torch.randperm(n_nodes, generator=torch.Generator().manual_seed(1))[:C].to(torch.int32)
        ns = torch.zeros(n_nodes, dtype=torch.uint8)
        for b, e, m in zip([0] + group_end[:-1], group_end, masks):
            ns[self.col_id[b:e].long()] = m
        self.node_splits = ns
        self._bank = torch.arange(C * D, dtype=torch.float32).view(C, D).to(torch.bfloat16)
        self.hier = hier

    def bank(self):
        return self._bank


@pytest.mark.parametrize("world", [1, 3, 8])
def test_split_shard_holds_its_slices(world):
    from hgrnet_b200.dist import SplitShard, split_shard_bounds
    se = _FakeSplitEval([10, 17, 40], [1, 3, 2], 100)
    rows = []
    for r in range(world):
        sh = SplitShard(se, r, world)
        ranges, local_end, kept = split_shard_bounds(se.group_end, world)[r]
        idx = torch.cat([torch.arange(lo, hi) for lo, hi in ranges]) if ranges else torch.zeros(0, dtype=torch.int64)
        assert torch.equal(sh.bank, se.bank()[idx]) and torch.equal(sh.col_id, se.col_id[idx])
        assert sh.group_end == local_end and sh.group_splits == [se.group_splits[g] for g in kept]
        assert sh.split_C == [17, 30] and sh.S == 2 and sh.names == ["s0", "s1"]
        assert sh.C == len(idx) and sh.D == 16 and sh.hier is None
        rows += idx.tolist()
    assert sorted(rows) == list(range(40))


@pytest.mark.parametrize("args,want", [((4096, 20, 8, 4, 1024), dict(slot_bytes=671744, x_off=2687232, total=36241664)),
                                       ((512, 20, 3, 4, 0), dict(slot_bytes=84144, total=336896))])
def test_exchange_layout_without_splits_is_unchanged(args, want):
    from hgrnet_b200.dist import exchange_layout
    lay = exchange_layout(*args)
    assert {k: lay[k] for k in want} == want
    assert exchange_layout(*args, n_splits=0) == lay
    assert exchange_layout(*args, n_levels=12, n_splits=0) == exchange_layout(*args, n_levels=12)


@pytest.mark.parametrize("B,K,world,S,n_levels", [(4096, 20, 8, 3, 0), (4096, 20, 8, 3, 12), (512, 20, 3, 2, 0),
                                                  (5, 20, 8, 8, 20), (33, 7, 3, 3, 32), (7, 1, 16, 1, 1)])
def test_exchange_layout_split_areas(B, K, world, S, n_levels):
    from hgrnet_b200.dist import exchange_layout
    base = exchange_layout(B, K, world, 4)
    lay = exchange_layout(B, K, world, 4, n_levels=n_levels, n_splits=S)
    area = 2 * world * base["part_bytes"] + (world * base["block_rows"] * 4 + 15) // 16 * 16   # lists, ids, bounds
    sb = lay["split_bytes"]
    assert sb % 16 == 0 and area <= sb < area + 16                       # aligned, and the areas of two splits disjoint
    assert lay["block_rows"] == base["block_rows"] and lay["part_bytes"] == base["part_bytes"]
    if n_levels:
        assert lay["hier_off"] == S * sb                                 # the winner words after the last split
        assert lay["slot_bytes"] >= lay["hier_off"] + world * lay["hier_part_bytes"]
    else:
        assert lay["slot_bytes"] == S * sb
    assert lay["slot_bytes"] % 16 == 0 and lay["total"] == (256 + 4 * lay["slot_bytes"] + 255) // 256 * 256
    if (B, K, world, S, n_levels) == (4096, 20, 8, 3, 0):
        assert abs(lay["slot_bytes"] - 2e6) < 0.05e6                     # ~2 MB per slot at cfg 5, G = 8, S = 3


def test_split_global_list_len_cfg5():
    """The per-split lists of a rank's part of the cfg-5 union bank under the global certificate: the 2-hops split sits
    in one or two lists per row and rank that hold 1/G of it, so G = 2 and 4 keep exact lists and G = 8 takes 16."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import split_shard_bounds
    got = {}
    for G in (2, 4, 8):
        lens = set()
        for ranges, local_end, kept in split_shard_bounds(CFG5_ENDS, G):
            masks = [CFG5_MASKS[g] for g in kept]
            lens.add(ops.splits_global_list_len(4096, local_end[-1], 1024, 20, local_end, masks, CFG5_SPLIT_C))
        assert len(lens) == 1                                            # every rank takes the same length
        got[G] = lens.pop()
    assert got == {2: 20, 4: 20, 8: 16}
    # one rank holding the whole union bank, and a single split: never narrower than the plain head's global policy
    assert ops.splits_global_list_len(4096, 20842, 1024, 20, CFG5_ENDS, CFG5_MASKS, CFG5_SPLIT_C) == 20
    assert ops.splits_global_list_len(4096, 2731, 1024, 20, [2731], [1], [21841]) >= ops.global_list_len(
        4096, 2731, 1024, 20, 21841)


def test_split_symbols_are_exported_and_tor_por_merged():
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    for name in ("hgr_score_topk_splits_scatter_bounded", "hgr_score_topk_splits_scatter_bounded_workspace_bytes",
                 "hgr_score_topk_splits_global_list_len", "hgr_topk_merge_splits_certified",
                 "hgr_hier_finish_rows_gathered", "hgr_hier_metrics_fused_rows"):
        assert hasattr(lib, name) and name in _cabi.SIGNATURES
    # one list set and several are the two modes of one TOR / POR entry point (node_splits, n_sets)
    for name in ("hgr_hier_finish_rows_gathered_splits", "hgr_hier_metrics_fused_rows_splits"):
        assert not hasattr(lib, name) and name not in _cabi.SIGNATURES
    assert len(_cabi.SIGNATURES["hgr_hier_finish_rows_gathered"][1]) == 19
    assert len(_cabi.SIGNATURES["hgr_hier_metrics_fused_rows"][1]) == 22
    assert lib.hgr_version() == 1


def test_merge_splits_certified_rejects_bad_arguments():
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    f = lib.hgr_topk_merge_splits_certified
    common = dict(P=2, B=4, K=20, S=3, ps=80, bs=4, ss=2 * 2 * 80 + 2 * 4)
    def call(**kw):
        a = dict(common, **kw)
        return f(16, 16, 16, a["P"], a["B"], a["K"], a["S"], a["ps"], a["bs"], a["ss"], None, 16, 10, 16, 16, None, 16,
                 64, 16, 1.0, None, None)
    assert call(P=0) == -1 and call(P=17) == -1                          # 1..16 shards
    assert call(S=0) == -1 and call(S=9) == -1                           # 1..8 splits
    assert call(K=33) == -1
    assert call(ps=79) == -1                                             # lists of two shards overlap
    assert call(bs=3) == -1
    assert call(ss=2 * 2 * 80 + 2 * 4 - 1) == -1                         # the areas of two splits overlap
    assert call(B=0) == 0                                                # nothing to merge: no launch


def test_scatter_rejects_bad_arguments():
    import ctypes
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    ends = (ctypes.c_int32 * 2)(10, 20)
    masks = (ctypes.c_uint8 * 2)(1, 3)
    ctot = (ctypes.c_int64 * 2)(20, 10)
    blocks = (ctypes.c_void_p * 2)(16, 16)
    def call(C=20, n_splits=2, n_groups=2, masks_=masks, ctot_=ctot, K=20, n_blocks=2, block_rows=2, ss=2 * 2 * 41):
        return lib.hgr_score_topk_splits_scatter_bounded(16, 16, None, 0, 4, C, 64, 1.0, K, n_groups, ends, masks_,
                                                         n_splits, ctot_, 16, 1 << 20, block_rows, n_blocks, blocks,
                                                         blocks, blocks, ss, 0, None)
    assert call(n_splits=9) == -1
    assert call(n_groups=17) == -1
    assert call(masks_=(ctypes.c_uint8 * 2)(1, 4)) == -1                 # a group names split 2 of two
    assert call(ctot_=None) == -1
    assert call(K=0) == -1
    assert call(n_blocks=17) == -1 and call(block_rows=1) == -1          # the blocks must cover B = 4 rows
    assert call(ss=2 * 2 * 41 - 1) == -1                                 # the areas of two splits overlap


def test_stream_rejects_bad_split_arguments():
    from hgrnet_b200.dist import HierShard, ShardedEvalStream, SplitShard
    se = _FakeSplitEval([10, 17, 40], [1, 3, 2], 100)
    sh = SplitShard(se, 0, 1)
    w = torch.zeros(40, 16, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="peer-memory"):
        ShardedEvalStream(w, 0, batch=64, steps=2, exchange="nccl", splits=sh)
    with pytest.raises(ValueError, match="certify='global'"):
        ShardedEvalStream(w, 0, batch=64, steps=2, certify="local", splits=sh)
    args = dict(bank_sorted=w, level_end=[40], sorted_to_pos=None, first_out=None, chain_ptr=None, chain_pos=None,
                chain_level=None)
    with pytest.raises(ValueError, match="hier"):
        ShardedEvalStream(w, 0, batch=64, steps=2, hier=HierShard(args, 0, 1), splits=sh)
    with pytest.raises(ValueError, match="banks"):
        ShardedEvalStream(w, 0, batch=64, steps=2, banks=[w, w], splits=sh)
    with pytest.raises(ValueError, match="D = 16"):
        ShardedEvalStream(torch.zeros(40, 32, dtype=torch.bfloat16), 0, batch=64, steps=2, splits=sh)
    with pytest.raises(ValueError, match="D = 16"):
        ShardedEvalStream(torch.zeros(40, 16, dtype=torch.bfloat16, device="meta"), 0, batch=64, steps=2, splits=sh)
