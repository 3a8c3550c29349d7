"""CPU tests of class-sharded TOR / POR (``hgr_hier_level_scatter`` / ``hgr_hier_finish_rows_gathered``): the cut of the
level-sorted train bank into shards, the exchange-slot layout, the library surface and the argument checks that fire
before any CUDA call."""
from __future__ import annotations

import ctypes

import pytest
import torch

HGR_ERR_BAD_ARG = -1


def _cut(level_end, world):
    from hgrnet_b200.dist import local_level_ends, shard_bounds
    M = level_end[-1]
    return [(lo, hi, local_level_ends(level_end, lo, hi)) for lo, hi in shard_bounds(M, world)]


@pytest.mark.parametrize("level_end,world", [([1, 21, 221], 8), ([3, 12, 52, 212], 3), ([0, 5, 5, 9, 40], 4),
                                             ([2, 2, 3], 8), ([1], 1), ([4096] * 3 + [5000], 5)])
def test_local_level_ends_cover_every_level(level_end, world):
    M = level_end[-1]
    level_of = [l for l, (a, b) in enumerate(zip([0] + level_end[:-1], level_end)) for _ in range(b - a)]
    assert len(level_of) == M
    seen = []
    for lo, hi, ends in _cut(level_end, world):
        assert len(ends) == len(level_end)
        assert ends == sorted(ends) and all(0 <= e <= hi - lo for e in ends)
        assert ends[-1] == hi - lo                                     # what the level GEMM requires
        starts = [0] + ends[:-1]
        for l, (a, b) in enumerate(zip(starts, ends)):
            assert all(level_of[lo + r] == l for r in range(a, b))      # local rows keep their global level
            seen += [lo + r for r in range(a, b)]
    assert seen == list(range(M))                                       # every sorted row in exactly one shard, in order


def test_local_level_ends_of_empty_shards():
    parts = _cut([1, 2, 3], 8)                                          # M = 3 < 8 ranks
    assert [hi - lo for lo, hi, _ in parts] == [1, 1, 1, 0, 0, 0, 0, 0]
    assert [ends for _, _, ends in parts[3:]] == [[0, 0, 0]] * 5
    assert [ends for _, _, ends in parts[:3]] == [[1, 1, 1], [0, 1, 1], [0, 0, 1]]


@pytest.mark.parametrize("args,want", [((4096, 20, 8, 4, 1024), dict(slot_bytes=671744, x_off=2687232, total=36241664)),
                                       ((512, 20, 3, 4, 0), dict(slot_bytes=84144, total=336896))])
def test_exchange_layout_without_levels_is_unchanged(args, want):
    from hgrnet_b200.dist import exchange_layout
    lay = exchange_layout(*args)
    assert set(lay) == {"block_rows", "part_bytes", "slot_bytes", "header", "x_off", "x_bytes", "total"}
    assert {k: lay[k] for k in want} == want
    assert exchange_layout(*args, n_levels=0) == lay


@pytest.mark.parametrize("B,K,world,D,n_levels", [(4096, 20, 8, 1024, 12), (512, 20, 3, 0, 20), (5, 20, 8, 0, 12),
                                                  (130, 20, 4, 64, 20), (33, 7, 3, 0, 32), (7, 1, 16, 0, 1)])
def test_exchange_layout_level_area(B, K, world, D, n_levels):
    from hgrnet_b200.dist import exchange_layout
    base = exchange_layout(B, K, world, 4, D)
    lay = exchange_layout(B, K, world, 4, D, n_levels)
    br = lay["block_rows"]
    assert lay["hier_off"] == base["slot_bytes"]                        # after the lists and bounds of the slot
    assert lay["hier_part_bytes"] == br * n_levels * 8
    assert lay["hier_off"] + world * lay["hier_part_bytes"] <= lay["slot_bytes"]
    assert lay["slot_bytes"] % 16 == 0 and lay["hier_off"] % 8 == 0
    for slot in range(4):                                               # every region of every slot 8-byte aligned
        start = lay["header"] + slot * lay["slot_bytes"] + lay["hier_off"]
        assert all((start + r * lay["hier_part_bytes"]) % 8 == 0 for r in range(world))
    assert lay["header"] + 4 * lay["slot_bytes"] <= lay["x_off"]        # slots stay clear of the feature replicas
    assert lay["total"] - lay["x_off"] == base["total"] - base["x_off"]


def test_hier_shard_holds_its_slice():
    from hgrnet_b200.dist import HierShard
    M, D = 23, 16
    bank = torch.arange(M * D, dtype=torch.float32).view(M, D).to(torch.bfloat16)
    args = dict(bank_sorted=bank, level_end=[1, 6, 23], sorted_to_pos=torch.arange(M, dtype=torch.int32),
                first_out=torch.tensor([1, 0, 0], dtype=torch.int32), chain_ptr=torch.zeros(2, dtype=torch.int32),
                chain_pos=torch.zeros(0, dtype=torch.int32), chain_level=torch.zeros(0, dtype=torch.int32))
    shards = [HierShard(args, r, 4) for r in range(4)]
    assert [(s.row_base, s.bank.shape[0]) for s in shards] == [(0, 6), (6, 6), (12, 6), (18, 5)]
    assert [s.level_end_local for s in shards] == [[1, 6, 6], [0, 0, 6], [0, 0, 6], [0, 0, 5]]
    assert all(s.M == M and s.D == D and s.n_levels == 3 and s.bank.is_contiguous() for s in shards)
    assert torch.equal(torch.cat([s.bank for s in shards]), bank)
    with pytest.raises(ValueError, match="32 levels"):
        HierShard(dict(args, level_end=list(range(1, 34))), 0, 2)


def test_new_symbols_are_exported():
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    for name in ("hgr_hier_level_scatter", "hgr_hier_finish_rows_gathered"):
        assert name in _cabi.SIGNATURES and hasattr(lib, name)


def _scatter_call(**kw):
    """hgr_hier_level_scatter with plausible fake device pointers (nothing is dereferenced: every case below must be
    refused before the first CUDA call)."""
    from hgrnet_b200 import _cabi
    a = dict(X=0x10000, bank=0x20000, B=64, M_r=40, D=128, ends=[10, 40], n_levels=2, row_base=0, ws=0x30000,
             ws_bytes=64 * 2 * 8, block_rows=16, dst=[0x40000 + 0x1000 * g for g in range(4)])
    a.update(kw)
    ends = (ctypes.c_int32 * max(1, len(a["ends"])))(*a["ends"])
    dst = (ctypes.c_void_p * max(1, len(a["dst"])))(*a["dst"])
    return _cabi.load().hgr_hier_level_scatter(a["X"], a["bank"], a["B"], a["M_r"], a["D"], ends, a["n_levels"],
                                                 a["row_base"], a["ws"], a["ws_bytes"], a["block_rows"], len(a["dst"]),
                                                 dst, None)


@pytest.mark.parametrize("bad", [dict(dst=[]), dict(dst=[0x40000 + 0x1000 * g for g in range(17)], block_rows=4),
                                 dict(block_rows=15), dict(n_levels=0), dict(n_levels=33), dict(row_base=-1),
                                 dict(row_base=(1 << 31) - 512), dict(dst=[0x40000, 0x41004, 0x42000, 0x43000]),
                                 dict(dst=[0x40000, 0, 0x42000, 0x43000]), dict(ws_bytes=64 * 2 * 8 - 1), dict(ws=None),
                                 dict(X=None), dict(bank=None), dict(X=0x10008), dict(D=100), dict(M_r=-1), dict(B=-1)])
def test_level_scatter_rejects_bad_arguments(bad):
    assert _scatter_call(**bad) == HGR_ERR_BAD_ARG


def test_level_scatter_empty_shard_needs_no_bank():
    # M_r == 0: X and the bank are not used, so null is fine there -- the next check (alignment of the workspace) fires
    assert _scatter_call(M_r=0, X=None, bank=None, ws=0x30004) == HGR_ERR_BAD_ARG
    from hgrnet_b200 import _cabi
    assert "workspace" in _cabi.load().hgr_last_error().decode()


def _finish_call(**kw):
    from hgrnet_b200 import _cabi
    a = dict(parts=0x10000, n_parts=4, stride=16 * 12, n_rows=16, M=500, n_levels=12, nodes=600, node_splits=None,
             n_sets=1)
    a.update(kw)
    p = 0x50000
    return _cabi.load().hgr_hier_finish_rows_gathered(a["parts"], a["n_parts"], a["stride"], a["n_rows"], a["M"],
                                                        a["n_levels"], p, p, p, a["nodes"], p, p, p, a["node_splits"],
                                                        a["n_sets"], None, None, p, None)


@pytest.mark.parametrize("bad", [dict(n_parts=0), dict(n_parts=17), dict(stride=16 * 12 - 1), dict(n_levels=0),
                                 dict(n_levels=33), dict(M=0), dict(nodes=0), dict(parts=None), dict(parts=0x10004),
                                 dict(n_rows=-1), dict(n_sets=0), dict(n_sets=2),
                                 dict(node_splits=0x60000, n_sets=0), dict(node_splits=0x60000, n_sets=9),
                                 dict(node_splits=0x60000, n_sets=3, n_rows=-1)])
def test_finish_gathered_rejects_bad_arguments_and_counter_sets(bad):
    assert _finish_call(**bad) == HGR_ERR_BAD_ARG


def test_finish_gathered_zero_rows_is_a_no_op_for_any_counter_sets():
    assert _finish_call(n_rows=0, parts=None) == 0
    assert _finish_call(n_rows=0, parts=None, node_splits=0x60000, n_sets=8) == 0
