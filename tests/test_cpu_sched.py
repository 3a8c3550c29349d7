"""The static schedule of the fused kernel (csrc/sched.cuh: chunks of (row tile, 16-row unit) space, the TileWalker
every CTA runs) checked exhaustively ON THE HOST: the header is plain integer arithmetic, so a small C++ harness
(tests/cpp/sched_check.cpp, built with g++) walks every worker of many shapes and verifies exact-once coverage,
sub-tile sizes, segment flags and the partial-list slot mapping the merge kernel relies on."""
from __future__ import annotations

import itertools
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
    exe = str(tmp_path_factory.mktemp("sched") / "sched_check")
    subprocess.run([gxx, "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "sched_check.cpp")],
                   check=True)
    return exe


def _run(exe, shapes):
    args = [str(v) for s in shapes for v in s]
    out = subprocess.run([exe] + args, capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout + out.stderr
    return int(out.stdout.split()[1])


def test_schedule_of_the_named_workloads(checker):
    shapes = []
    for (B, C) in [(64, 1000), (512, 21841), (256, 21841), (1024, 10450), (4096, 21841), (4096, 10921), (4096, 5461),
                   (4096, 2731), (512, 2731)]:
        for workers, rows in [(74, 256), (64, 256), (72, 256), (148, 128), (1, 256), (2, 128)]:
            shapes.append((B, C, workers, rows))
    assert _run(checker, shapes) == len(shapes)


def test_schedule_edge_and_random_shapes(checker):
    shapes = [(b, c, w, r) for b, c, w, r in itertools.product((1, 255, 256, 257, 513), (1, 15, 16, 17, 255, 256, 257, 4097),
                                                               (1, 3, 74), (128, 256))]
    rng = random.Random(0)
    for _ in range(400):
        shapes.append((rng.randint(1, 9000), rng.randint(1, 60000), rng.randint(1, 160), rng.choice((128, 256))))
    assert _run(checker, shapes) == len(shapes)
