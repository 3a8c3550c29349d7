"""Several test splits in one scoring pass on the class-sharded head (``hgr_score_topk_splits_scatter_bounded`` /
``hgr_topk_merge_splits_certified`` / ``hgr_hier_finish_rows_gathered`` with ``node_splits``, main.py:104-222 once per split): G
logical ranks inside one process on one GPU, as tests/test_gpu_peer.py does.  For every split the owners' result is
``ops.score_topk`` (exact lists) on that split's rows of the ranks' banks in rank-major order -- values, ids, order and
hits bit for bit when no owner repaired a row, rows always; then per-split TOR / POR, ``ShardedEvalStream(splits=...)`` against
``EvalStream(splits=...)``, and two real GPUs when the machine has them."""
from __future__ import annotations

import os
import socket

import numpy as np
import pytest
import torch

from tests.util import compare_topk, hits_from_idx, hostile_bank

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
K = 20


def _unit(n, d, seed):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    return (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)


class _Rows:
    """What ``SplitShard`` needs of an ``evaluate.HierMetrics``."""

    def __init__(self, args):
        self.args = args

    def rows_args(self):
        return self.args


class _Union:
    """What ``SplitShard`` needs of an ``evaluate.SplitEval``: the union bank of ``splits`` in group layout, built from
    ``rows`` (one bank row per node).  ``ordered``: the rows of every group in node order (hierarchy order) instead of
    the seeded permutation."""

    def __init__(self, splits, rows, ordered=False, hier_args=None):
        from hgrnet_b200.evaluate import split_groups
        n_nodes = rows.shape[0]
        self.names, nodes, self.group_end, self.group_splits, node_splits = split_groups(splits, n_nodes)
        if ordered:
            nodes = np.concatenate([np.sort(nodes[b:e]) for b, e in zip([0] + self.group_end[:-1], self.group_end)])
        self.S = len(self.names)
        self.col_id = torch.from_numpy(nodes).to(torch.int32).to(DEV)
        self.node_splits = torch.from_numpy(node_splits).to(DEV)
        self._bank = rows[torch.from_numpy(nodes)].to(DEV).contiguous()
        self.hier = _Rows(hier_args) if hier_args is not None else None

    def bank(self):
        return self._bank


def _run_sharded(u, x, targets, G, reps=1):
    """G logical ranks: every rank scatters its split lists and bounds, every owner certifies / repairs and counts.
    Returns (val [S, B, K], idx, counts [S, 6], per-split TOR / POR counters or None, repaired (row, split) pairs,
    the SplitShards)."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import PeerExchange, SplitShard, exchange_layout
    B = x.shape[0]
    shards = [SplitShard(u, r, G) for r in range(G)]
    n_levels = shards[0].hier.n_levels if u.hier is not None else 0
    lay = exchange_layout(B, K, G, 4, n_levels=n_levels, n_splits=u.S)
    bufs = [ops.peer_alloc(lay["total"])[0] for _ in range(G)]
    try:
        ranks = [PeerExchange(B, K, DEV, slots=4, _bases=bufs, _rank=r, _world=G, n_levels=n_levels, n_splits=u.S)
                 for r in range(G)]
        table = ops.shard_table([(sh.bank.data_ptr() if sh.C else 0, sh.col_id.data_ptr() if sh.C else 0, sh.C, 0)
                                 for sh in shards], DEV)
        counts = torch.zeros((u.S, ops.HGR_NUM_HITS + 1), dtype=torch.int64, device=DEV)
        hier_counts = ops.new_hier_counts(DEV, u.S) if n_levels else None
        repairs = torch.zeros(1, dtype=torch.int32, device=DEV)
        for rep in range(reps):
            slot = rep % 4
            for sh, px in zip(shards, ranks):
                px.scatter(x, sh.bank, 0, slot, col_id=sh.col_id, hier=sh.hier, splits=sh)
            outs = [px.merge(slot, targets, None, certify=(x, table, repairs), hier=sh.hier, counts=hier_counts,
                             splits=sh, split_counts=counts) for sh, px in zip(shards, ranks)]
        torch.cuda.synchronize()
        outs = [o for o in outs if o is not None]
        val = torch.cat([o[0] for o in outs], dim=1)
        idx = torch.cat([o[1] for o in outs], dim=1)
        return val, idx, counts.cpu(), hier_counts, int(repairs.item()), shards
    finally:
        torch.cuda.synchronize()
        for b in bufs:
            ops.peer_free(b)


def _rank_major(shards, s):
    """Split s's rows of the ranks' banks, rank after rank: (bank, node ids)."""
    banks, ids = [], []
    for sh in shards:
        rows = [torch.arange(b, e) for b, e, m in zip([0] + sh.group_end[:-1], sh.group_end, sh.group_splits)
                if (m >> s) & 1]
        if rows:
            r = torch.cat(rows).to(DEV)
            banks.append(sh.bank[r])
            ids.append(sh.col_id[r])
    return torch.cat(banks).contiguous(), torch.cat(ids).contiguous()


def _check(u, x, targets, G, reps=1, exact_ids=False):
    """Run G ranks and compare every split with ``score_topk`` on its rows in rank-major order.  The reference keeps
    exact lists, so its values are the GEMM's; without owner repairs the result must equal it bit for bit.  A repaired
    (row, split) carries CUDA-core values for its re-scanned shards: compared against the fp32 oracle, and with
    ``exact_ids`` (banks whose equal rows tie in either arithmetic) its ids and hits still bit for bit."""
    from hgrnet_b200 import ops
    val, idx, counts, _, repairs, shards = _run_sharded(u, x, targets, G, reps)
    in_all = u.node_splits[targets.long().clamp(min=0)] * (targets >= 0)
    for s in range(u.S):
        sub, sub_id = _rank_major(shards, s)
        in_s = ((in_all >> s) & 1).bool()
        t = torch.where(in_s, targets, torch.full_like(targets, -1))
        hits = ops.new_hits(DEV)
        v1, i1 = ops.score_topk(x, sub, col_id=sub_id, targets=t, hits=hits, impl=ops.HGR_IMPL_TCGEN05_EXACT)
        assert int(counts[s, ops.HGR_NUM_HITS]) == reps * int(in_s.sum()), "split %d rows" % s
        if repairs == 0 or exact_ids:
            assert torch.equal(idx[s], i1), "split %d: ids differ from score_topk in rank-major order" % s
            assert counts[s, :ops.HGR_NUM_HITS].tolist() == [reps * h for h in hits.tolist()], "split %d hits" % s
        if repairs == 0:
            assert torch.equal(val[s], v1), "split %d: values differ from score_topk in rank-major order" % s
        else:
            compare_topk(val[s], idx[s], (x.float() @ sub.float().T).cpu(), sub_id.cpu(), K)
        # the owner's counters are the Hit@k of the ids it returned (main.py:139-147), repaired rows included
        t_host = torch.where(t >= 0, t, torch.full_like(t, -2)).cpu()     # rows outside s: no id of a list matches
        assert counts[s, :ops.HGR_NUM_HITS].tolist() == [reps * h for h in hits_from_idx(idx[s], t_host)], \
            "split %d: hits differ from the returned ids" % s
    return repairs


def _splits(kind, nodes):
    """'hops': three nested sets of len * 1549/20842, len * 7860/20842 and all classes; 'overlap': three overlapping
    sets that are not nested (tests/test_gpu_eval_splits.py)."""
    C = len(nodes)
    if kind == "hops":
        a, b = max(1, C * 1549 // 20842), max(2, C * 7860 // 20842)
        return {"2-hops": nodes[:a], "3-hops": nodes[:b], "all": nodes}
    third = C // 3
    return {"a": nodes[:2 * third], "b": nodes[third:], "c": np.concatenate([nodes[:third // 2], nodes[-third // 2:]])}


def _case(kind, B, D, n_nodes, C, seed=0):
    from hgrnet_b200 import ops
    nodes = np.random.default_rng(seed).choice(n_nodes, size=C, replace=False)
    u = _Union(_splits(kind, nodes), _unit(n_nodes, D, 5))
    g = torch.Generator().manual_seed(7)
    targets = torch.from_numpy(nodes[torch.randint(0, C, (B,), generator=g).numpy()]).to(torch.int32).to(DEV)
    targets[3] = -1                                                       # a padded row: counted nowhere
    x = ops.normalize_rows(u.bank()[torch.randint(0, C, (B,), generator=g).to(DEV)].float()
                           + 0.5 * torch.randn(B, D, generator=g).to(DEV) / D ** 0.5)
    return u, x, targets


@pytest.mark.parametrize("kind", ["hops", "overlap"])
@pytest.mark.parametrize("G", [2, 8])
def test_cfg5_equals_score_topk_per_split(kind, G):
    u, x, targets = _case(kind, 4096, 1024, 21841, 20842)
    if kind == "hops":
        assert [e - b for b, e in zip([0] + u.group_end[:-1], u.group_end)] == [12982, 6311, 1549]
    assert _check(u, x, targets, G, reps=2) == 0


def test_b512_three_ranks():
    u, x, targets = _case("hops", 512, 512, 4000, 2900)
    _check(u, x, targets, 3, reps=3)                                      # 3 batches: slots reused


@pytest.mark.parametrize("G", [2, 5])
def test_split_with_fewer_than_k_classes(G):
    from hgrnet_b200 import ops
    nodes = np.random.default_rng(3).choice(3000, size=2000, replace=False)
    u = _Union({"tiny": nodes[:7], "all": nodes}, _unit(3000, 256, 5))
    x = ops.normalize_rows(torch.randn(300, 256, generator=torch.Generator().manual_seed(1)).to(DEV))
    targets = torch.from_numpy(nodes[np.arange(300) % 14]).to(torch.int32).to(DEV)
    _check(u, x, targets, G)
    val, idx, counts, _, _, _ = _run_sharded(u, x, targets, G)
    s = u.names.index("tiny")
    assert (idx[s, :, 7:] == -1).all() and torch.isinf(val[s, :, 7:]).all()
    assert int(counts[s, ops.HGR_NUM_HITS]) == sum(1 for i in range(300) if i % 14 < 7)   # labels of the tiny split


def test_groups_smaller_than_world_and_empty_ranks():
    """A group of 3 rows at G = 8 (five ranks hold none of it), and a union of 5 rows at G = 8 (four ranks hold no row
    at all): those ranks still store (-inf, -1) lists and -inf bounds, and the owners still merge."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import split_shard_bounds
    nodes = np.random.default_rng(4).choice(2000, size=1500, replace=False)
    rows = _unit(2000, 128, 5)
    x = ops.normalize_rows(torch.randn(200, 128, generator=torch.Generator().manual_seed(2)).to(DEV))
    targets = torch.from_numpy(nodes[np.arange(200) % 5]).to(torch.int32).to(DEV)
    u = _Union({"a": nodes[:3], "b": nodes}, rows)
    assert sorted(e - b for b, e in zip([0] + u.group_end[:-1], u.group_end)) == [3, 1497]
    _check(u, x, targets, 8)
    u = _Union({"a": nodes[:2], "b": nodes[2:5]}, rows)
    assert sum(1 for p in split_shard_bounds(u.group_end, 8) if not p[0]) == 4
    _check(u, x, targets, 8)


@pytest.mark.parametrize("kind", ["equal", "dups"])
@pytest.mark.parametrize("G", [3, 8])
def test_ties_across_every_shard_boundary(kind, G):
    """Equal bank rows everywhere: the order among equal values is (rank, local bank row), as score_topk on the ranks'
    banks concatenated rank after rank."""
    from hgrnet_b200 import ops
    nodes = np.random.default_rng(5).choice(3000, size=2400, replace=False)
    u = _Union(_splits("overlap", nodes), hostile_bank(3000, 256, kind))
    g = torch.Generator().manual_seed(8)
    x = ops.normalize_rows(u.bank()[torch.randint(0, 2400, (256,), generator=g).to(DEV)].float())
    targets = torch.from_numpy(nodes[torch.randint(0, 2400, (256,), generator=g).numpy()]).to(torch.int32).to(DEV)
    _check(u, x, targets, G, exact_ids=kind == "equal")


def test_clustered_bank_is_repaired_exactly():
    """Rows of every group in hierarchy order (siblings adjacent and similar) defeat the narrow lists: the owners must
    repair, and the result must still be the exact top-K of every split."""
    from hgrnet_b200 import ops
    nodes = np.random.default_rng(6).choice(22000, size=20842, replace=False)
    rows = hostile_bank(22000, 512, "clustered")
    u = _Union(_splits("hops", nodes), rows, ordered=True)
    g = torch.Generator().manual_seed(9)
    x = ops.normalize_rows(rows[torch.from_numpy(nodes[torch.randint(0, 20842, (4096,), generator=g).numpy()])].float()
                           .to(DEV) + 0.05 * torch.randn(4096, 512, generator=g).to(DEV) / 512 ** 0.5)
    targets = torch.from_numpy(nodes[torch.randint(0, 20842, (4096,), generator=g).numpy()]).to(torch.int32).to(DEV)
    assert _check(u, x, targets, 8) > 0, "a hierarchy-ordered bank should need owner repairs"


@pytest.mark.parametrize("split", ["all", "real"])
@pytest.mark.parametrize("G", [2, 8])
def test_per_split_tor_por_gathered_equal_single_gpu(split, G):
    from hgrnet_b200 import ops
    from tests.test_gpu_hier_sharded import _hierarchy, _rows_args, _split, _targets
    h = _hierarchy("cfg5")
    N, B, D = len(h), 4096, 1024
    bank = _unit(N, D, 21)
    args = _rows_args(h, _split(h, split), bank)
    nodes = np.random.default_rng(7).choice(N, size=20842, replace=False)
    u = _Union(_splits("hops", nodes), bank, hier_args=args)
    t = _targets(h, B, 50)
    t[:B // 2] = torch.from_numpy(nodes[np.arange(B // 2) % 3000]).to(torch.int32).to(DEV)   # rows in every split
    x = ops.normalize_rows(torch.randn(B, D, generator=torch.Generator().manual_seed(3)).to(DEV))
    _, _, _, hier_counts, _, _ = _run_sharded(u, x, t, G)
    want = ops.new_hier_counts(DEV, u.S)
    ops.hier_metrics_fused_rows(x, targets=t, node_splits=u.node_splits, counts=want, **args)
    assert torch.equal(hier_counts, want)
    assert all(int(want[s, :, 0].sum()) > 0 for s in range(u.S))


@pytest.mark.parametrize("host_io", [False, True])
def test_sharded_stream_single_rank_equals_eval_stream(tmp_path, host_io):
    """At world 1 the rank-major order is the union bank's order: ``ShardedEvalStream(splits=...)`` gives the counters and
    the top-K of ``EvalStream(splits=SplitEval)`` bit for bit."""
    from hgrnet_b200.dist import ShardedEvalStream, SplitShard
    from tests.test_gpu_eval_splits import _stream_model
    spec, model, h = _stream_model(tmp_path)
    N, B, steps = len(h), spec["B"], 4
    ids = np.random.default_rng(1).permutation(N)
    splits = {"small": ids[:30], "half": ids[:N // 2], "other": ids[N // 3:]}
    es = model.make_eval_stream(batch=B, slots=steps, streams=3, hier_metrics=True, eval_splits=splits)
    g = torch.Generator().manual_seed(6)
    feats = [torch.randn(B, spec["D"], generator=g) for _ in range(steps)]
    labels = [torch.from_numpy(ids[torch.randint(0, N, (B,), generator=g).numpy()]).to(torch.int32) for _ in range(steps)]
    labels[1][:10] = torch.from_numpy(ids[:10]).to(torch.int32)
    labels[2][0] = -1
    for s in range(steps):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for _ in range(2):
        for s in range(steps):
            es.step(s)
    es.end()
    se = es.splits
    ses = ShardedEvalStream(se.bank(), 0, batch=B, K=K, steps=steps, host_io=host_io, splits=SplitShard(se, 0, 1))
    for s in range(steps):
        (ses.host_feats if host_io else ses.dev_feats)[s].copy_(feats[s])
        (ses.host_labels if host_io else ses.dev_labels)[s].copy_(labels[s])
    ses.run()
    ses.run()
    torch.cuda.synchronize()
    for s in range(steps):
        assert torch.equal(ses.idx[s], es.idx[s]) and torch.equal(ses.val[s], es.val[s])
    assert ses.split_hit_counts() == es.split_hit_counts()
    assert ses.split_ratios() == es.split_ratios()
    assert int(ses.repairs.item()) == 0
    assert len(ses.split_lines()) == 3 and all(l.startswith(n + ": ") for l, n in zip(ses.split_lines(), se.names))
    if host_io:
        snaps = torch.stack(ses.host_counters)                   # the batch that finished last has seen every batch
        assert torch.equal(snaps.max(dim=0).values, ses.counters.cpu())
    ses.close()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        global DEV
        DEV = dev
        from hgrnet_b200 import ops
        from hgrnet_b200.dist import ShardedEvalStream, SplitShard
        u, x, targets = _case("hops", 512, 1024, 21841, 20842)
        feats = x.float()
        sh = SplitShard(u, rank, world)
        ses = ShardedEvalStream(u.bank(), 0, batch=512, K=K, steps=4, splits=sh)
        for s in range(4):
            ses.dev_feats[s].copy_(feats)
            ses.dev_labels[s].copy_(targets)
        ses.run()
        torch.cuda.synchronize()
        xn = ops.normalize_rows(feats)
        counts = torch.zeros((u.S, ops.HGR_NUM_HITS + 1), dtype=torch.int64, device=dev)
        ops.score_topk_splits(xn, targets=targets, counts=counts, bank=u.bank(), group_end=u.group_end,
                              group_splits=u.group_splits, n_splits=u.S, col_id=u.col_id, node_splits=u.node_splits)
        assert ses.split_hit_counts() == (4 * counts).tolist()
        lines = ses.split_lines()
        ses.close()
        out.put(("ok", rank, lines))
    except BaseException:  # noqa: BLE001 -- report, then leave without tearing NCCL down
        import traceback
        out.put(("fail", rank, traceback.format_exc()[-1500:]))
    finally:
        os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpus_match_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    stuck = False
    for p in procs:
        p.join(300)
        if p.exitcode is None:
            p.kill()
            stuck = True
    res = []
    while not out.empty():
        res.append(out.get())
    assert not stuck and len(res) == world and all(r[0] == "ok" for r in res), res
    assert res[0][2] == res[1][2]                               # split_lines() is the same on every rank
