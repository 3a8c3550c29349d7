"""Hierarchical mistake severity and LCA distance@k (``hgr_hier_mistakes`` / ``evaluate.MistakeMetrics``), host side: a
numpy / Python oracle written straight from ``c2p``, the depth-equals-index invariant it relies on (DAGs included),
hand-checked answers on a 3-level tree, the arithmetic of ``mistake_summary``, the C ABI's argument checks, the CLI
flag and ``dist.MistakeShard``'s row bounds at world size 2 over gloo.  The kernel is compared with this oracle in
tests/test_gpu_mistakes.py."""
from __future__ import annotations

import os
import random
import socket

import numpy as np
import pytest
import torch

HIT_CUTS = (1, 2, 5, 10, 20)
MAX_CHAIN = 32
N_COUNTERS = 2 + 2 * len(HIT_CUTS) + 2 * MAX_CHAIN + 2


def lca_dist(c2p, t, p):
    """(h, d) of label t and prediction p, from the definitions: chain(n) = c2p[n] + [n], depth(n) = len(c2p[n]), lca =
    the largest index where the two chains hold the same node (-1 without one), an id outside the nodes = the
    super-root."""
    dt = len(c2p[t])
    if not 0 <= p < len(c2p):
        return dt + 1, dt + 1
    ct, cp = list(c2p[t]) + [t], list(c2p[p]) + [p]
    lca = max([i for i in range(min(len(ct), len(cp))) if ct[i] == cp[i]], default=-1)
    return dt - lca, dt + len(c2p[p]) - 2 * lca


def oracle_counts(c2p, idx, targets, node_splits=None):
    """int64 ``[S, N_COUNTERS]`` counters of ``idx`` ([B, K] or [S, B, K] node ids) against ``targets`` [B]."""
    idx = np.asarray(idx)
    if idx.ndim == 2:
        idx = idx[None]
    S, B, K = idx.shape
    out = np.zeros((S, N_COUNTERS), dtype=np.int64)
    for r in range(B):
        t = int(targets[r])
        if not (0 <= t < len(c2p) and 1 <= len(c2p[t]) + 1 <= MAX_CHAIN):
            continue
        bits = 1 if node_splits is None else int(node_splits[t])
        for s in range(S):
            if not (bits >> s) & 1:
                continue
            hd = [lca_dist(c2p, t, int(p)) for p in idx[s, r]]
            c = out[s]
            c[0] += 1
            c[1] += int(idx[s, r, 0]) != t
            for i, k in enumerate(HIT_CUTS):
                c[2 + i] += sum(h for h, _ in hd[:k])
                c[7 + i] += sum(d for _, d in hd[:k])
            c[12 + min(hd[0][1], 2 * MAX_CHAIN + 1)] += 1
    return out


def _tree():
    from hgrnet_b200.hierarchy import ROOT, Hierarchy
    edges = [(ROOT, "a"), (ROOT, "b"), ("a", "a1"), ("a", "a2"), ("b", "b1"), ("a1", "a1x"), ("a1", "a1y"),
             ("a2", "a2x"), ("b1", "b1x")]
    h = Hierarchy([list(e) for e in edges])
    return h, h.index


def test_layout_length_matches_the_library():
    from hgrnet_b200 import _cabi
    assert _cabi.HGR_MISTAKE_COUNTERS == N_COUNTERS == 78


def test_known_answers_on_a_three_level_tree():
    h, ix = _tree()
    t = ix["a1x"]                                                   # depth 2
    want = {"a1x": (0, 0), "a1y": (1, 2), "a2x": (2, 4), "b1x": (3, 6), "a1": (1, 1), "a": (2, 2), "b": (3, 4)}
    for name, hd in want.items():
        assert lca_dist(h.c2p, t, ix[name]) == hd, name
    assert lca_dist(h.c2p, t, -1) == (3, 3)                         # empty entry: the super-root
    assert lca_dist(h.c2p, ix["a1"], ix["a1x"]) == (0, 1)            # a descendant of the label
    assert lca_dist(h.c2p, ix["a"], ix["b"]) == (1, 2)               # two roots: only the super-root is common
    # one row, K = 3: [sibling, cousin, empty]; label -1 and N are counted nowhere
    c = oracle_counts(h.c2p, [[ix["a1y"], ix["a2x"], -1]] * 3, [t, -1, len(h)])[0]
    assert c[:2].tolist() == [1, 1]
    assert c[2:7].tolist() == [1, 3, 6, 6, 6] and c[7:12].tolist() == [2, 6, 9, 9, 9]
    assert c[12 + 2] == 1 and c[12:].sum() == 1
    # a correct top-1: no mistake, d = 0 in the histogram
    c = oracle_counts(h.c2p, [[t, ix["a1"]]], [t])[0]
    assert c[:2].tolist() == [1, 0] and c[2:4].tolist() == [0, 1] and c[12] == 1


def _dag(seed):
    """The random multi-parent graphs of tests/test_cpu_oracle_and_host.py::test_dag_chains_equal_networkx_shortest_path."""
    from hgrnet_b200.hierarchy import ROOT, Hierarchy
    rnd = random.Random(seed)
    n = rnd.randint(30, 300)
    names = ["n%08d" % i for i in range(n)]
    edges = []
    for i, c in enumerate(names):
        cands = [ROOT] + names[:i]
        for p_ in rnd.sample(cands, min(rnd.choice([1, 1, 1, 2, 3]), len(cands))):
            edges.append([p_, c])
    rnd.shuffle(edges)
    return Hierarchy(edges)


def test_dag_depth_equals_index_and_chains_rejoin():
    """Every c2p[n] is a shortest root path, so chain entry i has depth i; on a DAG two chains may differ at some index
    and agree again deeper -- the LCA is the deepest agreement, not the end of the common prefix."""
    rejoin = 0
    for seed in range(12):
        h = _dag(seed)
        for n, c in enumerate(h.c2p):
            chain = list(c) + [n]
            assert [len(h.c2p[x]) for x in chain] == list(range(len(chain)))
            assert int(h.depth[n]) == len(c)
        rnd = random.Random(seed)
        for _ in range(400):
            t, p = rnd.randrange(len(h)), rnd.randrange(len(h))
            ct, cp = list(h.c2p[t]) + [t], list(h.c2p[p]) + [p]
            m = [i for i in range(min(len(ct), len(cp))) if ct[i] == cp[i]]
            prefix = next((i for i in range(min(len(ct), len(cp))) if ct[i] != cp[i]), min(len(ct), len(cp)))
            if m and m[-1] >= prefix:
                rejoin += 1
                hh, dd = lca_dist(h.c2p, t, p)
                assert hh == len(h.c2p[t]) - m[-1] and dd == len(h.c2p[t]) + len(h.c2p[p]) - 2 * m[-1]
    assert rejoin > 0, "no split-and-rejoin pair: the DAG case was not exercised"


def test_mistake_summary_arithmetic():
    from hgrnet_b200.evaluate import mistake_line, mistake_summary
    c = [0] * N_COUNTERS
    c[0], c[1] = 10, 4
    c[2:7] = [6, 14, 40, 90, 200]
    c[7:12] = [10, 30, 80, 170, 390]
    c[12], c[13], c[12 + 65] = 6, 3, 1
    s = mistake_summary(c)
    assert s["rows"] == 10 and s["mistakes"] == 4 and s["mistake_rate"] == 0.4
    assert s["severity_h"] == 6 / 4 and s["severity_d"] == 10 / 4
    assert [s["hdist@%d" % k] for k in HIT_CUTS] == [6 / 10, 14 / 20, 40 / 50, 90 / 100, 200 / 200]
    assert [s["dist@%d" % k] for k in HIT_CUTS] == [10 / 10, 30 / 20, 80 / 50, 170 / 100, 390 / 200]
    assert s["hist_d"][0] == 6 and s["hist_d"][-1] == 1 and len(s["hist_d"]) == 66
    s7 = mistake_summary(torch.tensor(c), K=7)                      # K < 20: divide by rows * min(k, K)
    assert s7["hdist@10"] == 90 / 70 and s7["hdist@20"] == 200 / 70 and s7["hdist@5"] == 40 / 50
    z = mistake_summary([0] * N_COUNTERS)
    assert z["mistake_rate"] == z["severity_h"] == z["hdist@1"] == 0.0
    assert mistake_line(s) == " mistake_rate(%):40.00 severity:1.50 hdist@1:0.60 hdist@5:0.80 hdist@20:1.00"
    with pytest.raises(ValueError):
        mistake_summary([0] * 5)


def test_flag_parses_and_is_off_by_default():
    from hgrnet_b200.flags import parse_args
    assert parse_args([]).hgr_mistake_metrics is False
    assert parse_args(["--hgr_mistake_metrics", "True"]).hgr_mistake_metrics is True
    o = parse_args(["--hgr_mistake_metrics", "True", "--hgr_eval_splits", "hops2,hops3,rest"])
    assert o.hgr_mistake_metrics is True and o.hgr_eval_splits == "hops2,hops3,rest"


def _abi(**kw):
    from hgrnet_b200 import _cabi
    a = dict(topk_idx=8, B=4, K=20, set_stride=80, n_sets=1, targets=8, node_splits=None, chain_ptr=8, chain_node=8,
             n_nodes=10, counts=8, stream=None)
    a.update(kw)
    return _cabi.load().hgr_hier_mistakes(*a.values())


@pytest.mark.parametrize("bad", [dict(K=0), dict(K=33), dict(B=-1), dict(n_nodes=0), dict(n_sets=2),
                                 dict(n_sets=9, node_splits=8), dict(n_sets=0), dict(n_sets=3, node_splits=8, set_stride=79),
                                 dict(topk_idx=None), dict(chain_node=None), dict(counts=None), dict(counts=12)])
def test_abi_rejects_bad_arguments(bad):
    assert _abi(**bad) == -1                                        # HGR_ERR_BAD_ARG, before any launch


def test_abi_zero_rows_is_a_no_op():
    assert _abi(B=0, topk_idx=None, targets=None, counts=None) == 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class _Chains:
    def __init__(self):
        self.chain_ptr = torch.zeros(3, dtype=torch.int32)
        self.chain_node = torch.zeros(2, dtype=torch.int32)


def _shard_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from hgrnet_b200.dist import MistakeShard, exchange_layout
        sh = MistakeShard(_Chains())                                    # rank / world from the process group
        assert (sh.rank, sh.world) == (rank, world)
        bounds = {}
        for B in (1, 2, 3, 37, 512, 4096):
            lo, hi = sh.row_bounds(B)
            br = exchange_layout(B, 20, world, 4)["block_rows"]        # PeerExchange's row blocks
            assert (lo, hi) == (min(B, rank * br), min(B, min(B, rank * br) + br))
            got = [None, None]
            dist.all_gather_object(got, (lo, hi))
            bounds[B] = got
        out.put((rank, bounds))
    finally:
        dist.destroy_process_group()


def test_mistake_shard_row_bounds_over_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    res = dict(out.get() for _ in range(2))
    assert res[0] == res[1]
    for B, ((lo0, hi0), (lo1, hi1)) in res[0].items():               # the two owners partition the batch
        assert lo0 == 0 and hi0 == lo1 and hi1 == B, (B, res[0][B])


def test_mistake_shard_rejects_a_rank_outside_the_world():
    from hgrnet_b200.dist import MistakeShard
    with pytest.raises(ValueError):
        MistakeShard(_Chains(), rank=2, world=2)
    assert MistakeShard(_Chains(), rank=0, world=1).row_bounds(37) == (0, 37)
