"""The grouped schedule of the multi-split head (csrc/sched.cuh: Groups, GroupWalker, group_slot*) checked exhaustively
ON THE HOST, like tests/test_cpu_sched.py does for the plain schedule: tests/cpp/sched_groups_check.cpp (g++) walks every
worker of many shapes and group tables and verifies exact-once coverage, that no segment crosses a group end, dense
column-ordered list slots, the column range / group recovered per slot, and that one group is the plain schedule."""
from __future__ import annotations

import os
import random
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path_factory.mktemp("sched_groups") / "sched_groups_check")
    subprocess.run([gxx, "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "sched_groups_check.cpp")],
                   check=True)
    return exe


def _run(exe, cases):
    args = []
    for B, workers, rows, ends in cases:
        args += [B, workers, rows, len(ends), *ends]
    out = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout + out.stderr
    return int(out.stdout.split()[1])


def _ends(sizes):
    out, c = [], 0
    for s in sizes:
        c += s
        out.append(c)
    return out


def test_grouped_schedule_of_the_named_workloads(checker):
    hops = _ends([1549, 7860 - 1549, 20842 - 7860])        # 2-hops / 3-hops / all, groups ordered by membership
    overlap = _ends([700, 900, 3000, 5000, 11000])
    cases = []
    for B in (64, 256, 512, 1024, 4096):
        for workers, rows in [(74, 256), (64, 256), (72, 256), (148, 128), (1, 256), (2, 128)]:
            for ends in ([20842], [21841], hops, overlap):
                cases.append((B, workers, rows, ends))
    assert _run(checker, cases) == len(cases)


def test_grouped_schedule_edge_tables(checker):
    rng = random.Random(1)
    cases = []
    for B in (1, 255, 256, 257, 513):
        for workers, rows in [(1, 128), (3, 256), (74, 256), (148, 128)]:
            cases.append((B, workers, rows, [1]))                              # one row in all
            cases.append((B, workers, rows, [1, 2, 3]))                          # groups of one row
            cases.append((B, workers, rows, [5, 17, 20, 300]))                   # fewer than K rows, unaligned ends
            cases.append((B, workers, rows, _ends([16] * 16)))                   # sixteen one-unit groups
            cases.append((B, workers, rows, _ends([rng.randint(1, 40) for _ in range(16)])))
    assert _run(checker, cases) == len(cases)


def test_group_ends_on_worker_boundaries(checker):
    # groups whose ends are multiples of 16 leave U = C / 16, so the chunk boundaries are known in advance: put group
    # ends exactly on them (a chunk start and a group start that coincide open ONE slot, not two)
    cases = []
    for B, C, workers, rows in [(512, 20480, 74, 256), (256, 4096, 16, 256), (1024, 2048, 148, 128), (300, 1600, 7, 128)]:
        U = C // 16
        MT = (B + rows - 1) // rows
        T = MT * U
        G = min(T, workers)
        bounds = sorted({w * T // G % U for w in range(1, G)} - {0})
        for pick in (bounds[:15], bounds[1::3][:15], bounds[-15:]):
            ends = [16 * b for b in pick] + [C]
            cases.append((B, workers, rows, ends))
            cases.append((B, workers, rows, [e + 1 for e in ends[:-1]] + [C]))   # one row past each boundary
    assert _run(checker, cases) == len(cases)


def test_grouped_schedule_random_tables(checker):
    rng = random.Random(0)
    cases = []
    for _ in range(400):
        n = rng.randint(1, 16)
        C = rng.randint(n, 30000)
        ends = sorted(rng.sample(range(1, C), n - 1)) + [C]
        cases.append((rng.randint(1, 5000), rng.randint(1, 160), rng.choice((128, 256)), ends))
    assert _run(checker, cases) == len(cases)
