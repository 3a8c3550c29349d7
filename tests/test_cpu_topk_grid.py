"""The shape grid of ``tests/test_gpu_topk_exact.py`` reaches what it claims, checked without a GPU through the
host-side plan (``ops.score_topk_plan`` / ``ops.global_list_len``; with no device visible the library assumes the
148 SMs of a B200) and a short restatement of the schedule (``sched.cuh``: ``make_sched`` / ``TileWalker``) and of the
merge dispatch (``topk_merge.cu``: ``launch_topk_merge``).  A policy change that drops a branch fails here."""
from __future__ import annotations

import pytest

from tests.test_gpu_topk_exact import EDGE_SHAPES, GRID

UNIT, SUB_N, CHUNK = 16, 256, 32          # sched.cuh kUnit / kSubN, umma_common.cuh kChunk
PAIRS = 74                                # CTA pairs of 148 SMs
ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    from hgrnet_b200 import ops as _ops
    ops = _ops


def exact_len(K):
    """List length of exact lists (score_launch.cu, pick_list_len without speculation)."""
    return 8 if K <= 8 else 12 if K <= 12 else 20 if K <= 20 else 32


def merge_kernel(P, KL):
    """Kernel ``launch_topk_merge`` picks for the scoring kernel's own lists (use_sched): by candidates per row."""
    cand = P * KL
    if cand <= 96:
        return "rank<2>" if cand <= 64 else "rank<3>"
    if cand <= 320:
        return "select<4>" if cand <= 128 else "select<6>" if cand <= 192 else "select<10>"
    return "merge<4>" if P <= 128 else "merge<10>"


def make_sched(B, C, workers, rows=2 * 128):
    MT, U = -(-B // rows), -(-C // UNIT)
    T = MT * U
    return dict(G=max(1, min(T, workers)), MT=MT, U=U, T=T)


def owner(s, x):
    return ((x + 1) * s["G"] - 1) // s["T"]


def parts(s, mt):
    return owner(s, (mt + 1) * s["U"] - 1) - owner(s, mt * s["U"]) + 1


def sub_tiles(s, C):
    """(n, nvalid) of every sub-tile of every worker (TileWalker::next)."""
    G, U, T = s["G"], s["U"], s["T"]
    for w in range(G):
        u, u_end = w * T // G, (w + 1) * T // G
        while u < u_end:
            mt, uu = divmod(u, U)
            nu = min(U - uu, u_end - u, SUB_N // UNIT)
            n = nu * UNIT
            yield n, min(n, C - uu * UNIT)
            u += nu


def _plan(B, C, D, K):
    return ops.score_topk_plan(B, C, D, K)


def _pairs(B, C, D, K):
    p = _plan(B, C, D, K)
    P, kl = p["lists_per_row"], p["list_len"]
    return {("production", kl, merge_kernel(P, kl)), ("exact", exact_len(K), merge_kernel(P, exact_len(K)))}


def test_restated_schedule_matches_the_plan():
    for B, C, D, K in GRID:
        p = _plan(B, C, D, K)
        s = make_sched(B, C, p["workers"])
        assert (s["G"], s["MT"], s["U"]) == (p["workers"], p["row_tiles"], p["units_per_row_tile"])
        assert max(parts(s, mt) for mt in range(s["MT"])) == p["lists_per_row"]
        assert -(-s["T"] // s["G"]) * UNIT == p["cols_per_worker"]


def test_grid_reaches_every_list_length_and_merge_kernel_pair():
    """Every (list length, merge kernel) pair the policy produces for production and for exact lists over a sweep of
    small shapes (K = 1..32; B decides the row tiles, C the lists per row; D does not enter the list-length rule)
    occurs on the grid, the speculative rank / select pairs included."""
    reach = set()
    for B in (1, 129, 257, 2047):
        for C in range(1, 1300, 7):
            for K in range(1, 33):
                reach |= _pairs(B, C, 64, K)
    got = set()
    for B, C, D, K in GRID:
        got |= _pairs(B, C, D, K)
    assert reach - got == set()
    for kl, kern in ((10, "rank<3>"), (10, "select<6>"), (16, "select<4>"), (16, "select<6>"), (16, "rank<2>"),
                     (8, "select<10>"), (10, "merge<4>")):
        assert ("production", kl, kern) in got
    assert {k for (_, _, k) in got} == {"rank<2>", "rank<3>", "select<4>", "select<6>", "select<10>", "merge<4>"}
    assert {K for (_, _, _, K) in GRID} >= {1, 7, 8, 9, 12, 13, 16, 20, 21, 32}


def test_grid_reaches_every_remainder_width_and_schedule_edge():
    widths, short, depths, aligned, B_set, D_set = set(), set(), set(), set(), set(), set()
    for B, C, D, K in GRID:
        p = _plan(B, C, D, K)
        s = make_sched(B, C, p["workers"])
        for n, nvalid in sub_tiles(s, C):
            widths.add(n)
            if nvalid < CHUNK and nvalid % UNIT:
                short.add(nvalid)
        depths.add(p["ring_depth"])
        # pick_sched: all pairs, or a multiple of the row tiles below that (no chunk straddles a row tile)
        aligned.add(p["workers"] < min(s["T"], PAIRS))
        B_set.add(B)
        D_set.add(D)
    assert widths == set(range(UNIT, SUB_N + 1, UNIT))
    assert short, "no sub-tile with fewer than 32 valid columns that is not a multiple of 16"
    assert depths == {4, 5}
    assert aligned == {True, False}
    assert B_set >= {1, 127, 128, 129, 255, 257} and min(B_set) < 2048 <= max(B_set) and 2047 in B_set
    assert D_set >= {8, 56, 64, 72, 1032}
    assert sum(B * C * D > 512 * 21841 * 1024 for B, C, D, _ in GRID) == 0
    assert sum(B >= 2048 for B, _, _, _ in GRID) <= 2


def test_grid_has_a_sketch_launch_with_solo_and_shared_row_tiles():
    """The sketch runs on all pairs (make_sched over 74); a row tile with one worker publishes no floor words."""
    mixed = []
    for B, C, D, K in GRID:
        s = make_sched(B, C, PAIRS)
        kinds = {parts(s, mt) == 1 for mt in range(s["MT"])}
        if K <= 20 and kinds == {True, False}:
            mixed.append((B, C))
    assert mixed


def test_edge_shapes_reach_every_merge_kernel():
    kernels = []
    for B, C, D, K in EDGE_SHAPES:
        p = _plan(B, C, D, K)
        assert p["lists_per_row"] >= 2
        kernels.append(merge_kernel(p["lists_per_row"], p["list_len"]))
    assert sorted(kernels) == sorted(["rank<2>", "rank<3>", "select<4>", "select<6>", "select<10>", "merge<4>"])


def test_global_list_lengths_of_the_certificate_test():
    assert {ops.global_list_len(1024, 2731, 256, 32, c) for c in (2731, 2 * 2731, 4 * 2731, 8 * 2731)} == {8, 10, 12, 16}
