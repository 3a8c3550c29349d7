"""Class-sharded TOR / POR (``hgr_hier_level_scatter`` / ``hgr_hier_finish_rows_gathered``, main.py:143,152-191): G
logical ranks inside one process on one GPU, as tests/test_gpu_peer.py does -- every rank runs the level GEMM on its
slice of the level-sorted train bank and pushes its winner words to the row owners, every owner finishes its rows --
against ``ops.hier_metrics_fused_rows`` on the whole batch, bit for bit; then inside ``ShardedEvalStream``, and over
two real GPUs when the machine has them."""
from __future__ import annotations

import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
K = 20


def _emb(n, d, seed, normalize=True):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    if normalize:
        x = x / x.norm(dim=-1, keepdim=True)
    return x.to(torch.bfloat16)


def _rows_args(h, train, bank):
    """What ``HierMetrics.rows_args()`` returns, built by hand as tests/test_gpu_hier_rows.py::_setup does: ``bank`` holds
    one row per node, ``train`` the train classes (train_index)."""
    from hgrnet_b200.evaluate import chain_table
    train_index = torch.tensor(train)
    depth = torch.from_numpy(h.depth).long()
    n_levels = int(depth.max()) + 1
    dt = depth[train_index]
    M = len(train)
    first_out = torch.tensor([int((dt != l).nonzero()[0]) if (dt != l).any() else M for l in range(n_levels)],
                             dtype=torch.int32, device=DEV)
    order = torch.sort(dt, stable=True).indices
    table = [torch.from_numpy(a).to(DEV) for a in chain_table(h.c2p, h.depth, train)]
    return dict(bank_sorted=bank[train_index][order].to(DEV).contiguous(),
                level_end=torch.cumsum(torch.bincount(dt, minlength=n_levels), 0).tolist(),
                sorted_to_pos=order.to(torch.int32).to(DEV), first_out=first_out,
                **dict(zip(("chain_ptr", "chain_pos", "chain_level"), table)))


def _targets(h, B, seed):
    """Random labels of every depth (depth 0 included, so L = 1 occurs); rows 1 and 3 are padding (-1 and N)."""
    N = len(h)
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, N, (B,), generator=g, dtype=torch.int32)
    for d in range(h.max_depth + 1):
        t[(5 + 7 * d) % B] = h.d2n[d][int(torch.randint(len(h.d2n[d]), (1,), generator=g))]
    if B > 3:
        t[1], t[3] = -1, N
    return t.to(DEV)


def _single(x, t, args):
    from hgrnet_b200 import ops
    B = x.shape[0]
    n_levels = len(args["level_end"])
    c = ops.new_hier_counts(DEV)
    lvl = torch.empty((B, n_levels), dtype=torch.int32, device=DEV)
    top1 = torch.empty((B,), dtype=torch.int32, device=DEV)
    ops.hier_metrics_fused_rows(x, targets=t, counts=c, lvl_idx=lvl, top1=top1, **args)
    return c, lvl, top1


def _run_sharded(batches, args, w, G, hier=True):
    """G logical ranks, plain (uncertified) list exchange plus, with ``hier``, the winner words.  ``batches`` = list of
    (x_norm, targets) run in turn through 4 slots.  Returns the owners' results of the LAST batch (val, idx, lvl_idx,
    top1 concatenated over owners), the hit counters and the owners' TOR / POR counters summed."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import HierShard, PeerExchange, exchange_layout, shard_bounds
    B = batches[0][0].shape[0]
    n_levels = len(args["level_end"]) if hier else 0
    lay = exchange_layout(B, K, G, 4, n_levels=n_levels)
    bufs = [ops.peer_alloc(lay["total"])[0] for _ in range(G)]
    try:
        ranks = [PeerExchange(B, K, DEV, slots=4, _bases=bufs, _rank=r, _world=G, n_levels=n_levels) for r in range(G)]
        shards = [HierShard(args, r, G) if hier else None for r in range(G)]
        cb = shard_bounds(w.shape[0], G)
        wsh = [w[lo:hi].contiguous() for lo, hi in cb]
        hits = ops.new_hits(DEV)
        counts = [ops.new_hier_counts(DEV) for _ in range(G)]
        for rep, (x, t) in enumerate(batches):
            slot = rep % 4
            for r, px in enumerate(ranks):
                px.scatter(x, wsh[r], cb[r][0], slot, hier=shards[r])
            outs = []
            for r, px in enumerate(ranks):
                n = px.hi - px.lo
                ho = None
                if hier and n > 0:
                    ho = (torch.full((n, n_levels), -7, dtype=torch.int32, device=DEV),
                          torch.full((n,), -7, dtype=torch.int32, device=DEV))
                o = px.merge(slot, t, hits, hier=shards[r], counts=counts[r], hier_out=ho)
                if o is not None:
                    outs.append((o, ho))
        torch.cuda.synchronize()
        val = torch.cat([o[0] for o, _ in outs])
        idx = torch.cat([o[1] for o, _ in outs])
        lvl = torch.cat([ho[0] for _, ho in outs]) if hier else None
        top1 = torch.cat([ho[1] for _, ho in outs]) if hier else None
        return val, idx, lvl, top1, hits, sum(c.cpu() for c in counts)
    finally:
        torch.cuda.synchronize()
        for b in bufs:
            ops.peer_free(b)


def _hierarchy(kind):
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    if kind == "cfg5":
        return synthetic_hierarchy(scaled_levels(21841), seed=1)
    if kind == "deep20":
        return synthetic_hierarchy([1 + i // 2 for i in range(20)], seed=3)
    if kind == "small":
        return synthetic_hierarchy([4, 20, 200], seed=3)
    return synthetic_hierarchy([1, 2], seed=3)                   # "tiny": 3 nodes, M < G


def _split(h, split):
    if split == "all":
        return list(range(len(h)))
    from tools.bench_hier_stream import real_split
    return real_split(h)


@pytest.mark.parametrize("kind,split,B,D,G", [("cfg5", "all", 4096, 1024, 8), ("cfg5", "all", 4096, 1024, 2),
                                             ("cfg5", "real", 4096, 1024, 8), ("cfg5", "real", 4096, 1024, 2),
                                             ("small", "all", 512, 256, 3), ("deep20", "all", 130, 64, 4),
                                             ("small", "all", 5, 128, 8), ("tiny", "all", 40, 64, 8)])
def test_sharded_equals_single_gpu(kind, split, B, D, G):
    h = _hierarchy(kind)
    N = len(h)
    train = _split(h, split)
    bank = _emb(N, D, 21)
    args = _rows_args(h, train, bank)
    M = len(train)
    if kind == "cfg5":
        assert len(args["level_end"]) == 12
    if kind == "tiny":
        assert M < G
    w = _emb(max(N, 300), D, 2).to(DEV)                          # the class bank of the lists
    from hgrnet_b200 import ops
    batches = [(ops.normalize_rows(_emb(B, D, 40 + i, normalize=False).float().to(DEV)), _targets(h, B, 50 + i))
               for i in range(3)]
    batches = [batches[i % 3] for i in range(6)]                 # 6 batches through 4 slots: every slot reused
    val, idx, lvl, top1, hits, counts = _run_sharded(batches, args, w, G)

    want = torch.zeros_like(counts)
    for x, t in batches:
        want += _single(x, t, args)[0].cpu()
    _, lvl1, top11 = _single(*batches[-1], args)
    assert torch.equal(lvl, lvl1), "per-level winners differ from the single-GPU call"
    assert torch.equal(top1, top11)
    assert torch.equal(counts, want), (counts[counts.any(1)], want[want.any(1)])
    assert int(want[:, 0].sum()) == 6 * (B - 2 if B > 3 else B)
    # the lists and Hit@k of the same run do not notice the winner words
    v0, i0, _, _, h0, _ = _run_sharded(batches, args, w, G, hier=False)
    assert torch.equal(val, v0) and torch.equal(idx, i0) and torch.equal(hits, h0)


@pytest.mark.parametrize("G", [3, 8])
def test_ties_across_shard_boundaries(G):
    """Equal bank rows on both sides of every shard boundary, and one level whose rows are all equal: the max over the
    shards' words must pick the first position, as the single-GPU epilogue does."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import shard_bounds
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    h = synthetic_hierarchy([3, 9, 40, 160], seed=3)             # level 2 = sorted rows [12, 52)
    N, D, B = len(h), 128, 256
    train = list(range(N))
    args = _rows_args(h, train, _emb(N, D, 21))
    bs = args["bank_sorted"]
    ends = args["level_end"]
    M = bs.shape[0]
    bounds = [lo for lo, _ in shard_bounds(M, G)[1:] if 0 < lo < M]
    for b in bounds:
        bs[b] = bs[b - 1]
    l_eq = 2                                                     # all of level 2 equal; at G = 8 it spans a boundary
    bs[ends[l_eq - 1]:ends[l_eq]] = bs[ends[l_eq - 1]]
    # queries: copies of the duplicated rows (they win their level, tied), then random rows
    src = torch.tensor(bounds + [ends[l_eq - 1]], device=DEV)
    x = ops.normalize_rows(_emb(B, D, 60, normalize=False).float().to(DEV))
    reps = src.repeat(B // (2 * len(src)) + 1)[:B // 2]
    x[:B // 2] = ops.normalize_rows(bs[reps].float())
    t = _targets(h, B, 61)
    _, _, lvl, top1, _, counts = _run_sharded([(x, t)], args, _emb(300, D, 2).to(DEV), G)
    c1, lvl1, top11 = _single(x, t, args)
    assert torch.equal(lvl, lvl1) and torch.equal(top1, top11) and torch.equal(counts, c1.cpu())
    # the ties were real: queries that copy the second row of an equal pair have the FIRST one as their top-1
    first = torch.tensor([b - 1 for b in bounds] + [ends[l_eq - 1]], device=DEV)
    first = first.repeat(B // (2 * len(src)) + 1)[:B // 2]
    pos = args["sorted_to_pos"].long()
    assert bool((top1[:B // 2].long() == pos[first]).any())


class _Rows:
    """What ``EvalStream(hier=...)`` needs of an ``evaluate.HierMetrics``."""

    def __init__(self, args):
        self.args = args

    def rows_args(self):
        return self.args


@pytest.mark.parametrize("host_io", [False, True])
def test_sharded_eval_stream_single_rank_counter_block(host_io):
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import HierShard, ShardedEvalStream
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    from hgrnet_b200.stream import EvalStream
    h = synthetic_hierarchy([5, 45, 400, 4550], seed=3)
    N, B, D = len(h), 300, 512
    w = _emb(N, D, 2).to(DEV)
    args = _rows_args(h, list(range(0, N, 3)), w.cpu())
    feats = [torch.randn(B, D, generator=torch.Generator().manual_seed(10 + s)) for s in range(8)]
    labels = [_targets(h, B, 30 + s).cpu() for s in range(8)]
    streams = {}
    for mode in ("off", "on"):
        ses = ShardedEvalStream(w, 0, batch=B, K=K, steps=8, host_io=host_io,
                                hier=HierShard(args, 0, 1) if mode == "on" else None)
        for s in range(8):
            (ses.host_feats if host_io else ses.dev_feats)[s].copy_(feats[s])
            (ses.host_labels if host_io else ses.dev_labels)[s].copy_(labels[s])
        ses.run()
        ses.run()
        streams[mode] = ses
    torch.cuda.synchronize()
    off, on = streams["off"], streams["on"]
    for s in range(8):
        assert torch.equal(on.val[s], off.val[s]) and torch.equal(on.idx[s], off.idx[s])
    assert torch.equal(on.hits, off.hits)
    want = ops.new_hier_counts(DEV)
    for s in range(8):
        ops.hier_metrics_fused_rows(ops.normalize_rows(feats[s].to(DEV)), targets=labels[s].to(DEV), counts=want, **args)
    assert torch.equal(on.hier_counts[0], 2 * want)
    if host_io:
        snaps = torch.stack(on.host_counters)                    # the batch that finished last has seen every batch
        assert torch.equal(snaps.max(dim=0).values, on.counters.cpu())
        assert torch.equal(torch.stack(on.host_hits).max(dim=0).values, on.hits.cpu())
    es = EvalStream(w, batch=B, slots=8, streams=3, host_io=False, hier=_Rows(args))
    for s in range(8):
        es.dev_feats[s].copy_(feats[s])
        es.dev_labels[s].copy_(labels[s])
    es.begin()
    for _ in range(2):
        for s in range(8):
            es.step(s)
    es.end()
    assert on.hier_ratios() == es.hier_ratios()
    assert es.hit_counts() == on.all_reduce_hits().tolist()
    assert all(r > 0 for r in on.hier_ratios())
    for ses in streams.values():
        ses.close()


def test_rejected_inputs():
    from hgrnet_b200.dist import HierShard, ShardedEvalStream
    h = _hierarchy("small")
    N = len(h)
    args = _rows_args(h, list(range(N)), _emb(N, 128, 21))
    w = _emb(N, 128, 2).to(DEV)
    with pytest.raises(ValueError, match="peer-memory"):
        ShardedEvalStream(w, 0, batch=64, steps=2, exchange="nccl", hier=HierShard(args, 0, 1))
    with pytest.raises(ValueError, match="32 levels"):
        HierShard(dict(args, level_end=list(range(1, 34))), 0, 1)
    with pytest.raises(ValueError, match="D = 128"):
        ShardedEvalStream(_emb(N, 64, 2).to(DEV), 0, batch=64, steps=2, hier=HierShard(args, 0, 1))


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
        from hgrnet_b200.dist import HierShard, ShardedEvalStream, shard_bounds
        h = _hierarchy("cfg5")
        N, B, D = len(h), 512, 1024
        w = _emb(N, D, 2)
        args = _rows_args(h, _split(h, "real"), w)
        feats = torch.randn(B, D, generator=torch.Generator().manual_seed(9))
        t = _targets(h, B, 10)
        lo, hi = shard_bounds(N, world)[rank]
        ses = ShardedEvalStream(w[lo:hi].to(dev).contiguous(), lo, batch=B, K=K, steps=8, hier=HierShard(args, rank, world))
        for s in range(8):
            ses.dev_feats[s].copy_(feats.to(dev))
            ses.dev_labels[s].copy_(t)
        ses.run()
        ses.run()
        torch.cuda.synchronize()
        x = ops.normalize_rows(feats.to(dev))
        c1, _, _ = _single(x, t, args)
        h1 = ops.new_hits(dev)
        rv, ri = ops.score_topk(x, w.to(dev), targets=t, K=K, hits=h1)
        c = ses.hier_counts[0].clone()
        dist.all_reduce(c)
        assert torch.equal(c, 16 * c1), "all-reduced TOR / POR counters differ from the single-GPU call"
        assert ses.all_reduce_hits().tolist() == [16 * v for v in h1.tolist()]
        for s in (0, 7):
            assert torch.equal(ses.idx[s], ri[ses.row_lo:ses.row_hi]) and torch.equal(ses.val[s], rv[ses.row_lo:ses.row_hi])
        ratios = ses.hier_ratios()
        assert all(r > 0 for r in ratios)
        ses.close()
        out.put(("ok", rank, ratios))
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
    assert res[0][2] == res[1][2]                               # hier_ratios() is the same on every rank
