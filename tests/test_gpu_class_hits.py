"""Per-class Hit@k on the device (``hgr_class_hits``), integer for integer: the table equals the oracle of
tests/test_cpu_class_hits.py on the head's own top-K lists at the cfg-2 shape (per-row labels, one label for the whole
batch, padding, labels outside the bank, K < 20, C < K, several list sets with overlapping masks); summed over classes
it equals the Hit@k / per-split counters the scoring calls keep today; the eager ``test()`` line with and without
``--hgr_class_metrics``; ``EvalStream`` against eager ``ClassHits``; and the class-sharded owners / ``ShardedEvalStream``
against one GPU."""
from __future__ import annotations

import os
import socket

import numpy as np
import pytest
import torch

from tests.test_cpu_class_hits import oracle_class_counts

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
K = 20
N, C, B, D = 21841, 20842, 512, 1024          # cfg 2: 21,841 nodes, 20,842 test classes, B = 512


def _unit(n, d, seed):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    return (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)


def _check(idx, targets, n_nodes, node_splits=None):
    """Run the kernel on ``idx`` and compare the table with the oracle, counter by counter; returns the table."""
    from hgrnet_b200 import ops
    S = idx.shape[0] if idx.dim() == 3 else 1
    counts = ops.new_class_counts(DEV, n_nodes, S)
    ops.class_hits(idx, targets, counts, node_splits=node_splits)
    want = oracle_class_counts(idx.cpu().numpy(), targets.cpu().numpy(), n_nodes,
                               None if node_splits is None else node_splits.cpu().numpy())
    got = counts.cpu().numpy()
    assert np.array_equal(got, want), np.argwhere(got != want)[:10]
    return got


@pytest.fixture(scope="module")
def cfg2():
    """The cfg-2 bank (test classes = 20,842 of the 21,841 nodes, node ids as col_id) and its node table."""
    rows = _unit(N, D, 3).to(DEV)
    nodes = np.sort(np.random.default_rng(0).choice(N, size=C, replace=False))
    col_id = torch.from_numpy(nodes).to(torch.int32).to(DEV)
    return rows, rows[col_id.long()].contiguous(), col_id, nodes


def _near(rows, near, seed):
    """Normalised features close to ``rows[near]``, with a noise that grows along the batch: the label lands at every
    position of the list, and past it."""
    from hgrnet_b200 import ops
    g = torch.Generator().manual_seed(seed)
    n = len(near)
    noise = torch.linspace(0.2, 12.0, n)[torch.randperm(n, generator=g)].to(DEV)[:, None]
    return ops.normalize_rows(rows[near].float() + noise * torch.randn(n, D, generator=g).to(DEV) / D ** 0.5)


def _labels(kind, nodes, seed):
    g = torch.Generator().manual_seed(seed)
    pick = lambda ids, n: torch.from_numpy(ids[torch.randint(0, len(ids), (n,), generator=g).numpy()])
    if kind == "one_label":
        t = torch.full((B,), int(nodes[123]), dtype=torch.int64)
    elif kind == "outside_bank":                                        # rows count, hits never
        t = pick(np.setdiff1d(np.arange(N), nodes), B)
    else:
        t = pick(nodes, B)
        t[1], t[3] = -1, N                                              # padding: counted nowhere
        if kind == "padding":
            t[::2] = -1
            t[1::4] = N
    return t.to(torch.int32).to(DEV)


@pytest.mark.parametrize("kind", ["random", "one_label", "padding", "outside_bank"])
def test_kernel_equals_oracle_on_score_topk_lists(cfg2, kind):
    from hgrnet_b200 import ops
    rows, bank, col_id, nodes = cfg2
    t = _labels(kind, nodes, 4)
    near = t.long().clamp(0, N - 1)
    x = _near(rows, near, 5)
    _, idx = ops.score_topk(x, bank, col_id=col_id, K=K)
    got = _check(idx, t, N)[0]
    counted = int(((t >= 0) & (t < N)).sum())
    assert got[:, -1].sum() == counted
    if kind == "outside_bank":
        assert got[:, :-1].sum() == 0
    else:
        assert 0 < got[:, 0].sum() < got[:, 4].sum() <= counted        # the labels sit at many positions
    if kind == "one_label":
        assert got[int(t[0]), -1] == B and got[:, -1].sum() == B
    for k in (7, 3):                                                    # K < 20: only the first K entries exist
        _check(ops.score_topk(x, bank, col_id=col_id, K=k)[1], t, N)


def test_fewer_classes_than_k(cfg2):
    """K = 7 against a bank of 5 classes: entries 5 and 6 are empty (-1) and match no label."""
    from hgrnet_b200 import ops
    rows, _, _, nodes = cfg2
    cls = torch.from_numpy(nodes[[5, 300, 301, 9000, 20000]]).to(torch.int32).to(DEV)
    x = _near(rows, cls[torch.arange(64, device=DEV) % 5].long(), 7)
    t = cls[torch.arange(64, device=DEV) % 5].clone()
    t[::3] = int(nodes[6])
    t[1] = -1
    _, idx = ops.score_topk(x, rows[cls.long()].contiguous(), col_id=cls, K=7)
    assert (idx[:, 5:] == -1).all()
    got = _check(idx, t, N)[0]
    assert got[:, 0].sum() > 0


def _union(kind, nodes):
    from tests.test_gpu_splits_sharded import _Union, _splits
    return _Union(_splits(kind, nodes), _unit(N, D, 3))


@pytest.mark.parametrize("kind", ["hops", "overlap"])
def test_split_lists_equal_oracle_and_split_counts(cfg2, kind):
    """``[S, B, K]`` lists of ``score_topk_splits`` with nested and overlapping split masks: the table equals the
    oracle, and summed over classes the split's ``[Hit@1 .. Hit@20, rows]`` counters of the scoring call itself."""
    from hgrnet_b200 import ops
    rows, _, _, nodes = cfg2
    u = _union(kind, nodes)
    t = _labels("random", nodes, 8)
    x = _near(rows, t.long().clamp(0, N - 1), 9)
    counts = torch.zeros((u.S, ops.HGR_NUM_HITS + 1), dtype=torch.int64, device=DEV)
    _, idx = ops.score_topk_splits(x, u.bank(), u.group_end, u.group_splits, u.S, col_id=u.col_id, targets=t,
                                   node_splits=u.node_splits, counts=counts)
    got = _check(idx, t, N, u.node_splits)
    assert np.array_equal(got.sum(1), counts.cpu().numpy())
    assert all(c[0] > 0 for c in counts.tolist())
    _check(idx[:, 64:192], t[64:192].contiguous(), N, u.node_splits)   # a row slice of each set (set_stride > B * K)
    _check(torch.randint(-1, N, (u.S, B, K), dtype=torch.int32, device=DEV), t, N, u.node_splits)


def test_table_sums_to_score_topk_hits(cfg2):
    from hgrnet_b200 import ops
    rows, bank, col_id, nodes = cfg2
    t = _labels("random", nodes, 10)
    x = _near(rows, t.long().clamp(0, N - 1), 11)
    hits = ops.new_hits(DEV)
    _, idx = ops.score_topk(x, bank, col_id=col_id, targets=t, K=K, hits=hits)
    got = _check(idx, t, N)[0]
    assert got[:, :-1].sum(0).tolist() == hits.tolist() and got[:, -1].sum() == B - 2


# ---- eager test() -----------------------------------------------------------------------------------------------
def _lines(model, batches, flag, splits=None):
    from hgrnet_b200 import evaluate
    from hgrnet_b200.synthetic import FeatureLoader
    opts = model.opts
    opts.print_freq, opts.hgr_class_metrics = 1000, flag
    opts.hgr_eval_splits = ",".join(splits) if splits else ""
    return evaluate.test(opts, model, DEV, loader=FeatureLoader([f for f, _ in batches], [l for _, l in batches]),
                         splits=None if splits is None else {k: [model.nodes[i] for i in v] for k, v in splits.items()},
                         log=False).strip()


@pytest.mark.parametrize("with_splits", [False, True])
def test_eager_test_line(tmp_path, with_splits):
    """``test()`` with the flag prints the oracle's class-averaged values after today's line (after each split's line
    with ``--hgr_eval_splits``); without it, exactly today's line."""
    from oracle import cases
    from tests.test_gpu_hier_rows import _model
    from hgrnet_b200.evaluate import SplitEval, class_line, class_summary
    spec = cases.EVAL_CASES[0]
    model, h, test_ids = _model(spec, tmp_path)
    n = len(h)
    g = torch.Generator().manual_seed(11)
    batches = [(torch.randn(spec["B"], spec["D"], generator=g), int(test_ids[(7 * b) % len(test_ids)]))
               for b in range(6)]
    splits = None
    if with_splits:
        ids = sorted(set(int(i) for i in test_ids))
        splits = {"s0": ids[:len(ids) // 2], "s1": ids[len(ids) // 4:], "all": ids}
    off = _lines(model, batches, False, splits)
    on = _lines(model, batches, True, splits)
    assert "class_mean" not in off
    se = SplitEval(model, splits, hier=False) if with_splits else None
    want = 0
    with torch.no_grad():
        for f, l in batches:
            x = model.encode_image_normalized(f.to(DEV))
            t = torch.full((f.shape[0],), l, dtype=torch.int32, device=DEV)
            if se is None:
                idx, ns = model.score_topk(None, t, feats_normalized=x)[1], None
            else:
                idx, ns = se.update(x, t)[1], se.node_splits.cpu().numpy()
            want = want + oracle_class_counts(idx.cpu().numpy(), t.cpu().numpy(), n, ns)
    off_lines, on_lines = off.split("\n"), on.split("\n")
    assert len(on_lines) == len(off_lines) == (3 if with_splits else 1)
    for s, (a, b) in enumerate(zip(off_lines, on_lines)):
        assert b == a + class_line(class_summary(want[s]))
    if with_splits:
        assert class_summary(want[0])["classes"] > 0


# ---- EvalStream ---------------------------------------------------------------------------------------------------
def _stream_batches(h, spec, steps, ids):
    n, b = len(h), spec["B"]
    g = torch.Generator().manual_seed(6)
    feats = [torch.randn(b, spec["D"], generator=g) for _ in range(steps)]
    labels = [torch.from_numpy(ids[torch.randint(0, n, (b,), generator=g).numpy()]).to(torch.int32) for _ in range(steps)]
    labels[1][:10] = torch.from_numpy(ids[:10]).to(torch.int32)
    labels[2][0] = -1
    labels[3][:] = int(ids[0])                                          # a one-class batch, as the reference's loader
    return feats, labels


def _replay(es, feats, labels, reps, steps):
    for s in range(steps):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for _ in range(reps):
        for s in range(steps):
            es.step(s)
    es.end()


@pytest.mark.parametrize("with_splits", [False, True])
def test_eval_stream_equals_eager(tmp_path, with_splits):
    from hgrnet_b200.evaluate import ClassHits, SplitEval, class_summary
    from tests.test_gpu_eval_splits import _stream_model
    spec, model, h = _stream_model(tmp_path)
    n, steps = len(h), 4
    ids = np.random.default_rng(1).permutation(n)
    splits = {"small": ids[:30], "half": ids[:n // 2], "other": ids[n // 3:]} if with_splits else None
    es = model.make_eval_stream(batch=spec["B"], slots=steps, streams=3, eval_splits=splits, class_metrics=True)
    plain = model.make_eval_stream(batch=spec["B"], slots=steps, streams=3, eval_splits=splits)
    assert es.host_counters.numel() == plain.host_counters.numel()    # the table is not in the per-step copy
    feats, labels = _stream_batches(h, spec, steps, ids)
    _replay(es, feats, labels, 3, steps)
    if with_splits:
        eager = SplitEval(model, splits, hier=False, class_metrics=True)
        for s in range(steps):
            eager.update(model.encode_image_normalized(feats[s].to(DEV)), labels[s].to(DEV))
        want = 3 * eager.classes.counts.cpu()
        assert torch.equal(es.class_table(), want)
        assert es.split_class_summary() == [class_summary(c) for c in want]
        assert all(l.count(" class_mean Top@1(%):") == 1 for l in eager.lines())
        with pytest.raises(RuntimeError):
            es.class_summary()
    else:
        ch = ClassHits(model)
        for s in range(steps):
            x = model.encode_image_normalized(feats[s].to(DEV))
            ch.update(model.score_topk(None, labels[s].to(DEV), feats_normalized=x)[1], labels[s].to(DEV))
        want = 3 * ch.table()
        assert torch.equal(es.class_table(), want)
        assert int(want[:, -1].sum()) == 3 * (steps * spec["B"] - 1)
        assert es.class_summary() == class_summary(want)
        with pytest.raises(RuntimeError):
            es.split_class_summary()


# ---- class-sharded ------------------------------------------------------------------------------------------------
def _owner_table(idx, t, G, n_nodes, node_splits=None):
    """Every owner counts its rows of the merged lists (``ShardedEvalStream``'s rule); the tables summed."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import exchange_layout
    S = idx.shape[0] if idx.dim() == 3 else 1
    br = exchange_layout(t.numel(), K, G, 4)["block_rows"]
    counts = ops.new_class_counts(DEV, n_nodes, S)
    for r in range(G):
        lo, hi = min(t.numel(), r * br), min(t.numel(), r * br + br)
        if hi > lo:
            ops.class_hits(idx[..., lo:hi, :], t[lo:hi].contiguous(), counts, node_splits=node_splits)
    return counts


@pytest.mark.parametrize("bank_kind,G,with_splits", [("iid", 2, False), ("iid", 8, False), ("clustered", 8, False),
                                                     ("iid", 2, True), ("iid", 8, True), ("clustered", 8, True)])
def test_sharded_owners_equal_one_gpu(bank_kind, G, with_splits):
    from hgrnet_b200 import ops
    from tests.util import hostile_bank
    b = 1024
    rows = _unit(N, D, 5).to(DEV) if bank_kind == "iid" else hostile_bank(N, D, "clustered").to(DEV)
    nodes = np.random.default_rng(6).choice(N, size=C, replace=False)
    g = torch.Generator().manual_seed(9)
    t = torch.from_numpy(nodes[torch.randint(0, C, (b,), generator=g).numpy()]).to(torch.int32).to(DEV)
    t[5] = -1
    t[100:164] = t[100]                                                 # one label over two whole warps
    x = ops.normalize_rows(rows[t.long().clamp(min=0)].float() + 0.05 * torch.randn(b, D, generator=g).to(DEV) / D ** 0.5)
    if with_splits:
        from tests.test_gpu_splits_sharded import _Union, _run_sharded, _splits
        u = _Union(_splits("hops", nodes), rows.cpu(), ordered=bank_kind != "iid")
        _, idx, _, _, repairs, _ = _run_sharded(u, x, t, G)
        _, idx1 = ops.score_topk_splits(x, u.bank(), u.group_end, u.group_splits, u.S, col_id=u.col_id)
        ns = u.node_splits
    else:
        from tests.test_gpu_hier_sharded import _run_sharded
        _, idx, _, _, _, _ = _run_sharded([(x, t)], None, rows, G, hier=False)
        _, idx1 = ops.score_topk(x, rows, K=K)
        ns, repairs = None, None
    got = _owner_table(idx, t, G, N, ns)
    want = oracle_class_counts(idx.cpu().numpy(), t.cpu().numpy(), N, None if ns is None else ns.cpu().numpy())
    assert np.array_equal(got.cpu().numpy(), want)
    one = ops.new_class_counts(DEV, N, got.shape[0])
    ops.class_hits(idx1, t, one, node_splits=ns)
    if with_splits and bank_kind == "clustered":
        assert repairs > 0, "a hierarchy-ordered bank should need owner repairs"
    if torch.equal(idx, idx1.view_as(idx)):
        assert torch.equal(got, one)
    else:                       # a repaired list or an exact tie may order equal-looking entries differently
        assert torch.equal(got[..., -1], one[..., -1])


@pytest.mark.parametrize("with_splits", [False, True])
def test_sharded_stream_single_rank_equals_eval_stream(tmp_path, with_splits):
    from hgrnet_b200.dist import ShardedEvalStream, SplitShard
    from hgrnet_b200.evaluate import ClassHits, EvalCounters
    from tests.test_gpu_eval_splits import _stream_model
    spec, model, h = _stream_model(tmp_path)
    n, b, steps = len(h), spec["B"], 4
    ids = np.random.default_rng(1).permutation(n)
    splits = {"small": ids[:30], "half": ids[:n // 2], "other": ids[n // 3:]} if with_splits else None
    es = model.make_eval_stream(batch=b, slots=steps, streams=3, eval_splits=splits, class_metrics=True)
    feats, labels = _stream_batches(h, spec, steps, ids)
    _replay(es, feats, labels, 2, steps)
    host_io = with_splits                                               # the host-fed owner path too
    if with_splits:
        se = es.splits
        ses = ShardedEvalStream(se.bank(), 0, batch=b, K=K, steps=steps, splits=SplitShard(se, 0, 1),
                                classes=ClassHits(model), host_io=True)
        assert ses.host_counters[0].numel() == EvalCounters(DEV, n_splits=se.S).counters.numel()
    else:
        ses = ShardedEvalStream(model.bank_test, 0, batch=b, K=K, steps=steps, col_id=model._test_index_i32,
                                classes=ClassHits(model))
        with pytest.raises(ValueError):
            ShardedEvalStream(model.bank_test, 0, batch=b, K=K, steps=steps, col_id=model._test_index_i32,
                              exchange="nccl", classes=ClassHits(model))
    for s in range(steps):
        (ses.host_feats if host_io else ses.dev_feats)[s].copy_(feats[s])
        (ses.host_labels if host_io else ses.dev_labels)[s].copy_(labels[s])
    ses.run()
    ses.run()
    torch.cuda.synchronize()
    table = ses.class_table()
    if not with_splits:
        assert int(table[:, -1].sum()) == 2 * (steps * b - 1)
    if all(torch.equal(ses.idx[s], es.idx[s]) for s in range(steps)):
        assert torch.equal(table, es.class_table())
    if with_splits:
        assert ses.split_class_summary() == es.split_class_summary() or not torch.equal(ses.idx[0], es.idx[0])
        assert all(" class_mean Top@1(%):" in l for l in ses.split_lines())
    else:
        assert ses.class_summary() == es.class_summary() or not torch.equal(ses.idx[0], es.idx[0])
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
        import tests.test_gpu_splits_sharded as tss
        global DEV
        DEV = tss.DEV = dev
        from hgrnet_b200 import ops
        from hgrnet_b200.dist import ShardedEvalStream, SplitShard
        u, x, targets = tss._case("hops", 512, 1024, N, C)
        classes = type("C", (), dict(n_nodes=N, counts=ops.new_class_counts(dev, N, 1)))()
        ses = ShardedEvalStream(u.bank(), 0, batch=512, K=K, steps=4, splits=SplitShard(u, rank, world),
                                classes=classes)
        for s in range(4):
            ses.dev_feats[s].copy_(x.float())
            ses.dev_labels[s].copy_(targets)
        ses.run()
        torch.cuda.synchronize()
        _, idx = ops.score_topk_splits(ops.normalize_rows(x.float()), u.bank(), u.group_end, u.group_splits, u.S,
                                       col_id=u.col_id)
        one = ops.new_class_counts(dev, N, u.S)
        ops.class_hits(idx, targets, one, node_splits=u.node_splits)
        got = ses.class_table()
        assert torch.equal(got, 4 * one.cpu())
        ses.close()
        out.put(("ok", rank, int(got[..., -1].sum())))
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
