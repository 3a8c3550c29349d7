"""The schedule on a share of the grid (``HGR_IMPL_GRID_SHARE``) and the policy that picks the share, checked without a
GPU through the host-side plan (``ops.score_topk_plan(grid_share=...)``, ``ops.score_topk_grid_share``; with no device
visible the library assumes the 148 SMs of a B200) and the schedule harness of ``tests/test_cpu_sched.py``."""
from __future__ import annotations

import random

import pytest

from tests.test_cpu_sched import _run, checker  # noqa: F401  (the fixture builds the harness)

PAIRS = 74   # CTA pairs of 148 SMs
ROWS = 256   # image rows per row tile (one CTA pair)
ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    from hgrnet_b200 import ops as _ops
    ops = _ops


SHAPES = [(512, 21841, 1024), (1024, 10450, 512), (4096, 21841, 1024), (2048, 21841, 1024), (256, 21841, 1024),
          (64, 1000, 1024), (1, 300, 64), (257, 4097, 1032), (1999, 5003, 56), (9500, 20, 64)]


def _plans():
    rng = random.Random(1)
    shapes = SHAPES + [(rng.randint(1, 9000), rng.randint(1, 60000), 8 * rng.randint(1, 160)) for _ in range(60)]
    return [(B, C, D, c, ops.score_topk_plan(B, C, D, 20, grid_share=c)) for B, C, D in shapes for c in (2, 3, 4, 8)]


def test_a_share_takes_its_budget_of_pairs_in_whole_row_tiles():
    for B, C, D, c, p in _plans():
        MT, T = -(-B // ROWS), -(-B // ROWS) * -(-C // 16)
        budget = max(1, PAIRS // c)
        want = budget // MT * MT if budget >= MT else budget
        assert p["row_tiles"] == MT
        assert p["workers"] == min(want, T), (B, C, c, p)
        if p["workers"] >= MT and T >= want:
            assert p["workers"] % MT == 0, (B, C, c, p)
            assert p["lists_per_row"] == p["workers"] // MT, (B, C, c, p)


def test_a_shared_schedule_covers_every_unit_exactly_once(checker):  # noqa: F811
    shapes = [(B, C, p["workers"], ROWS) for B, C, D, c, p in _plans()]
    assert _run(checker, shapes) == len(shapes)


def test_policy_keeps_the_whole_grid_on_long_streams():
    assert ops.score_topk_grid_share(4096, 21841, 1024) == 1                 # cfg 5
    for B in (2048, 3000, 4096, 8192):
        for C in (300, 2731, 10450, 21841, 60000):
            assert ops.score_topk_grid_share(B, C, 1024) == 1, (B, C)
    for B, C in ((1024, 60000), (1536, 60000)):                               # > 3,072 columns per worker
        assert ops.score_topk_plan(B, C, 1024)["cols_per_worker"] > 3072
        assert ops.score_topk_grid_share(B, C, 1024) == 1, (B, C)
    assert ops.score_topk_grid_share(512, 21841, 1024, 40) == 1              # K > 32: no tcgen05 kernel


def test_policy_and_plan_at_cfg2():
    """cfg 2 shares the grid two ways: 36 pairs, 18 per row tile, ~1,214 columns per worker; the list-length rule,
    applied to the longer lists (share 1 / 18.5 of a row's columns each), moves from 8 to 10 entries."""
    assert ops.score_topk_grid_share(512, 21841, 1024) == 2
    assert ops.score_topk_grid_share(1024, 10450, 512) == 2                   # cfg 4
    full = ops.score_topk_plan(512, 21841, 1024)
    half = ops.score_topk_plan(512, 21841, 1024, grid_share=2)
    assert (full["workers"], full["lists_per_row"], full["list_len"]) == (74, 37, 8)
    assert (half["workers"], half["lists_per_row"], half["list_len"], half["cols_per_worker"]) == (36, 18, 10, 1216)
    assert ops.score_topk_plan(512, 21841, 1024, grid_share=1) == full == ops.score_topk_plan(512, 21841, 1024,
                                                                                             grid_share=0)


def test_workspace_covers_every_share():
    from hgrnet_b200 import _cabi
    lib = _cabi.load()
    for B, C, D, c, p in _plans():
        K = 20
        lists = p["lists_per_row"] * B * 20 * 8   # exact lists of 20 (value, id) entries, the most a share can ask
        assert lib.hgr_score_topk_workspace_bytes(B, C, D, K) >= lists, (B, C, c, p)


def test_out_of_range_shares_are_refused():
    from hgrnet_b200 import _cabi
    with pytest.raises(_cabi.HgrError):
        ops.score_topk_plan(512, 21841, 1024, grid_share=9)
    with pytest.raises(_cabi.HgrError):
        ops.score_topk_plan(512, 21841, 1024, grid_share=-1)
