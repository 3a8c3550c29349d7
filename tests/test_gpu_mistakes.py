"""Hierarchical mistake severity and LCA distance@k on the device (``hgr_hier_mistakes``): the counters equal the oracle
of tests/test_cpu_mistakes.py exactly on the head's own top-K lists (cfg 1, the 21,841-node hierarchy, a DAG, K < 20
and C < K, overlapping splits, padded rows); the eager ``test()`` line with and without ``--hgr_mistake_metrics``;
``EvalStream`` against eager ``MistakeMetrics``; and ``ShardedEvalStream`` / the owners' merged lists against one GPU."""
from __future__ import annotations

import os
import socket

import numpy as np
import pytest
import torch

from tests.test_cpu_mistakes import _dag, oracle_counts

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
K = 20


def _unit(n, d, seed):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    return (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)


def _table(c2p):
    from hgrnet_b200.evaluate import chain_csr
    ptr, nodes = chain_csr(c2p)
    return dict(chain_ptr=torch.from_numpy(ptr.astype(np.int32)).to(DEV),
                chain_node=torch.from_numpy(nodes.astype(np.int32)).to(DEV))


def _check(c2p, idx, targets, node_splits=None):
    """Run the kernel on ``idx`` and compare with the oracle, counter by counter; returns the counters."""
    from hgrnet_b200 import ops
    S = idx.shape[0] if idx.dim() == 3 else 1
    counts = ops.new_mistake_counts(DEV, S)
    ops.hier_mistakes(idx, targets, counts=counts, node_splits=node_splits, **_table(c2p))
    want = oracle_counts(c2p, idx.cpu().numpy(), targets.cpu().numpy(),
                         None if node_splits is None else node_splits.cpu().numpy())
    got = counts.cpu().numpy()
    assert np.array_equal(got, want), np.argwhere(got != want)[:10]
    return got


def _near(bank, rows, noise, seed):
    """Normalised features close to bank rows ``rows`` (many right and many near-miss predictions)."""
    from hgrnet_b200 import ops
    g = torch.Generator().manual_seed(seed)
    D = bank.shape[1]
    return ops.normalize_rows(bank[rows].float() + noise * torch.randn(len(rows), D, generator=g).to(DEV) / D ** 0.5)


def _labels(N, B, seed):
    t = torch.randint(0, N, (B,), generator=torch.Generator().manual_seed(seed), dtype=torch.int32)
    t[1], t[3] = -1, N                                                   # padding: counted nowhere
    return t.to(DEV)


@pytest.mark.parametrize("kind", ["21841", "dag"])
def test_kernel_equals_oracle_on_score_topk_lists(kind):
    from hgrnet_b200 import ops
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    if kind == "21841":
        h, B, D = synthetic_hierarchy(scaled_levels(21841), seed=1), 512, 1024
    else:
        h, B, D = max((_dag(s) for s in range(12)), key=lambda x: x.n_multipath), 300, 128
    N = len(h)
    bank = _unit(N, D, 3).to(DEV)
    t = _labels(N, B, 4)
    near = t.long().clamp(0, N - 1)
    near[1::2] = torch.randint(0, N, (B // 2,), generator=torch.Generator().manual_seed(6)).to(DEV)   # other nodes
    x = _near(bank, near, 1.0, 5)
    _, idx = ops.score_topk(x, bank, K=K)
    c = _check(h.c2p, idx, t)
    assert c[0, 0] == B - 2 and 0 < c[0, 1] < B - 2                        # padding skipped; hits and mistakes
    assert c[0, 12] > 0 and c[0, 13:].sum() > 0


def test_kernel_equals_oracle_on_the_head_cfg1(tmp_path):
    from oracle import cases
    from tests.test_gpu_hier_rows import _model
    from hgrnet_b200.evaluate import MistakeMetrics
    spec = cases.EVAL_CASES[0]
    model, h, test_ids = _model(spec, tmp_path)
    B = 256
    t = torch.from_numpy(np.asarray(test_ids)[np.arange(B) % len(test_ids)]).to(torch.int32).to(DEV)
    t[7] = -1
    x = model.encode_image_normalized(torch.randn(B, spec["D"], generator=torch.Generator().manual_seed(2)).to(DEV))
    _, idx = model.score_topk(None, t, feats_normalized=x)
    mm = MistakeMetrics(model)
    mm.update(idx, t)
    mm.update(idx, t)
    want = oracle_counts(h.c2p, idx.cpu().numpy(), t.cpu().numpy())
    assert np.array_equal(mm.counts.cpu().numpy(), 2 * want)


def test_short_lists_and_fewer_classes_than_k():
    """K = 7 against a bank of 5 classes: entries 5 and 6 are empty (-1) and count as the super-root."""
    from hgrnet_b200 import ops
    from hgrnet_b200.hierarchy import synthetic_hierarchy
    h = synthetic_hierarchy([4, 20, 200], seed=3)
    N = len(h)
    cls = torch.tensor([5, 30, 31, 100, 200], dtype=torch.int32, device=DEV)
    bank = _unit(N, 64, 6).to(DEV)
    x = _near(bank, cls[torch.arange(64, device=DEV) % 5].long(), 2.0, 7)
    t = _labels(N, 64, 8)
    t[::4] = cls[0]
    val, idx = ops.score_topk(x, bank[cls.long()].contiguous(), col_id=cls, K=7)
    assert (idx[:, 5:] == -1).all()
    _check(h.c2p, idx, t)
    _check(h.c2p, ops.score_topk(x, bank, K=3)[1], t)


def test_splits_with_overlapping_masks():
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    h = synthetic_hierarchy(scaled_levels(21841), seed=1)
    N, B, S = len(h), 512, 3
    g = torch.Generator().manual_seed(9)
    idx = torch.randint(-1, N, (S, B, K), generator=g, dtype=torch.int32).to(DEV)
    t = _labels(N, B, 10)
    idx[:, :100, 0] = t[:100]                                            # some right top-1s
    node_splits = torch.randint(0, 8, (N,), generator=g).to(torch.uint8).to(DEV)   # any overlap
    c = _check(h.c2p, idx, t, node_splits)
    assert all(c[s, 0] > 0 for s in range(S))
    _check(h.c2p, idx[:, 64:192], t[64:192].contiguous(), node_splits)   # a row slice of each set (set_stride > B * K)


def _lines(model, batches, flag):
    from hgrnet_b200 import evaluate
    from hgrnet_b200.synthetic import FeatureLoader
    opts = model.opts
    opts.print_freq, opts.hgr_mistake_metrics = 1000, flag
    return evaluate.test(opts, model, DEV, loader=FeatureLoader([f for f, _ in batches], [l for _, l in batches]),
                         log=False).strip()


def test_eager_test_line(tmp_path):
    """``test()`` with the flag prints the oracle's values after today's line; without it, exactly today's line."""
    from oracle import cases
    from tests.test_gpu_hier_rows import _model
    from hgrnet_b200.evaluate import mistake_line, mistake_summary
    spec = cases.EVAL_CASES[0]
    model, h, test_ids = _model(spec, tmp_path)
    g = torch.Generator().manual_seed(11)
    batches = [(torch.randn(spec["B"], spec["D"], generator=g), int(test_ids[(7 * b) % len(test_ids)]))
               for b in range(4)]
    off = _lines(model, batches, False)
    on = _lines(model, batches, True)
    assert "mistake_rate" not in off and on.startswith(off + " mistake_rate(%):")
    want = np.zeros(oracle_counts(h.c2p, np.zeros((1, 1), np.int32), [-1]).shape[1], dtype=np.int64)
    with torch.no_grad():
        for f, l in batches:
            x = model.encode_image_normalized(f.to(DEV))
            t = torch.full((f.shape[0],), l, dtype=torch.int32, device=DEV)
            _, idx = model.score_topk(None, t, feats_normalized=x)
            want += oracle_counts(h.c2p, idx.cpu().numpy(), t.cpu().numpy())[0]
    assert on == off + mistake_line(mistake_summary(want))


def _stream_batches(h, spec, steps, ids):
    N, B = len(h), spec["B"]
    g = torch.Generator().manual_seed(6)
    feats = [torch.randn(B, spec["D"], generator=g) for _ in range(steps)]
    labels = [torch.from_numpy(ids[torch.randint(0, N, (B,), generator=g).numpy()]).to(torch.int32) for _ in range(steps)]
    labels[1][:10] = torch.from_numpy(ids[:10]).to(torch.int32)
    labels[2][0] = -1
    return feats, labels


@pytest.mark.parametrize("with_splits", [False, True])
def test_eval_stream_equals_eager(tmp_path, with_splits):
    from hgrnet_b200.evaluate import MistakeMetrics, SplitEval, mistake_summary
    from tests.test_gpu_eval_splits import _stream_model
    spec, model, h = _stream_model(tmp_path)
    N, steps = len(h), 4
    ids = np.random.default_rng(1).permutation(N)
    splits = {"small": ids[:30], "half": ids[:N // 2], "other": ids[N // 3:]} if with_splits else None
    es = model.make_eval_stream(batch=spec["B"], slots=steps, streams=3, eval_splits=splits, mistake_metrics=True)
    feats, labels = _stream_batches(h, spec, steps, ids)
    for s in range(steps):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for _ in range(3):
        for s in range(steps):
            es.step(s)
    es.end()
    es.synchronize()
    if with_splits:
        eager = SplitEval(model, splits, hier=False, mistakes=True)
        for s in range(steps):
            eager.update(model.encode_image_normalized(feats[s].to(DEV)), labels[s].to(DEV))
        assert torch.equal(es.mistake_counts, 3 * eager.mistakes.counts)
        assert es.split_mistake_summary() == [mistake_summary(c) for c in 3 * eager.mistakes.counts]
        assert all(l.count(" mistake_rate(%):") == 1 for l in eager.lines())
    else:
        mm = MistakeMetrics(model)
        for s in range(steps):
            x = model.encode_image_normalized(feats[s].to(DEV))
            mm.update(model.score_topk(None, labels[s].to(DEV), feats_normalized=x)[1], labels[s].to(DEV))
        assert torch.equal(es.mistake_counts, 3 * mm.counts)
        assert int(es.mistake_counts[0, 0]) == 3 * (steps * spec["B"] - 1)
        with pytest.raises(RuntimeError):
            es.split_mistake_summary()


def _sharded_counts(u, x, t, G, c2p):
    """G logical ranks on one GPU (tests/test_gpu_splits_sharded.py): every owner counts its merged rows as
    ``ShardedEvalStream`` does.  Returns (summed counters, merged idx [S, B, K], repairs)."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import MistakeShard
    from tests.test_gpu_splits_sharded import _run_sharded
    _, idx, _, _, repairs, _ = _run_sharded(u, x, t, G)
    tab = _table(c2p)
    counts = ops.new_mistake_counts(DEV, u.S)
    for r in range(G):
        lo, hi = MistakeShard(type("M", (), tab)(), r, G).row_bounds(x.shape[0])
        if hi > lo:
            ops.hier_mistakes(idx[:, lo:hi], t[lo:hi].contiguous(), counts=counts, node_splits=u.node_splits, **tab)
    return counts, idx, repairs


@pytest.mark.parametrize("bank_kind,G", [("iid", 2), ("iid", 8), ("clustered", 8)])
def test_sharded_owners_equal_one_gpu(bank_kind, G):
    from hgrnet_b200 import ops
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    from tests.test_gpu_splits_sharded import _Union, _splits
    from tests.util import hostile_bank
    h = synthetic_hierarchy(scaled_levels(21841), seed=1)
    N, B, D = len(h), 1024, 512
    nodes = np.random.default_rng(6).choice(N, size=20842, replace=False)
    rows = _unit(N, D, 5) if bank_kind == "iid" else hostile_bank(N, D, "clustered")
    u = _Union(_splits("hops", nodes), rows, ordered=bank_kind != "iid")
    g = torch.Generator().manual_seed(9)
    t = torch.from_numpy(nodes[torch.randint(0, 20842, (B,), generator=g).numpy()]).to(torch.int32).to(DEV)
    t[5] = -1
    x = ops.normalize_rows(rows[t.long().clamp(min=0).cpu()].float().to(DEV)
                           + 0.05 * torch.randn(B, D, generator=g).to(DEV) / D ** 0.5)
    counts, idx, repairs = _sharded_counts(u, x, t, G, h.c2p)
    one = ops.new_mistake_counts(DEV, u.S)
    _, idx1 = ops.score_topk_splits(x, u.bank(), u.group_end, u.group_splits, u.S, col_id=u.col_id)
    ops.hier_mistakes(idx1, t, counts=one, node_splits=u.node_splits, **_table(h.c2p))
    assert np.array_equal(counts.cpu().numpy(),
                          oracle_counts(h.c2p, idx.cpu().numpy(), t.cpu().numpy(), u.node_splits.cpu().numpy()))
    if bank_kind == "clustered":
        assert repairs > 0, "a hierarchy-ordered bank should need owner repairs"
    if torch.equal(idx, idx1):
        assert torch.equal(counts, one)
    else:                       # a repaired list or an exact tie may order equal-looking entries differently
        assert torch.equal(counts[:, :1], one[:, :1])


@pytest.mark.parametrize("with_splits", [False, True])
def test_sharded_stream_single_rank_equals_eval_stream(tmp_path, with_splits):
    from hgrnet_b200.dist import MistakeShard, ShardedEvalStream, SplitShard
    from hgrnet_b200.evaluate import MistakeMetrics
    from tests.test_gpu_eval_splits import _stream_model
    spec, model, h = _stream_model(tmp_path)
    N, B, steps = len(h), spec["B"], 4
    ids = np.random.default_rng(1).permutation(N)
    splits = {"small": ids[:30], "half": ids[:N // 2], "other": ids[N // 3:]} if with_splits else None
    es = model.make_eval_stream(batch=B, slots=steps, streams=3, eval_splits=splits, mistake_metrics=True)
    feats, labels = _stream_batches(h, spec, steps, ids)
    for s in range(steps):
        es.host_feats[s].copy_(feats[s])
        es.host_labels[s].copy_(labels[s])
    es.begin()
    for _ in range(2):
        for s in range(steps):
            es.step(s)
    es.end()
    ms = MistakeShard(MistakeMetrics(model), 0, 1)
    if with_splits:
        se = es.splits
        ses = ShardedEvalStream(se.bank(), 0, batch=B, K=K, steps=steps, splits=SplitShard(se, 0, 1), mistakes=ms)
    else:
        ses = ShardedEvalStream(model.bank_test, 0, batch=B, K=K, steps=steps, col_id=model._test_index_i32,
                                mistakes=ms)
    for s in range(steps):
        ses.dev_feats[s].copy_(feats[s])
        ses.dev_labels[s].copy_(labels[s])
    ses.run()
    ses.run()
    torch.cuda.synchronize()
    if all(torch.equal(ses.idx[s], es.idx[s]) for s in range(steps)):
        assert torch.equal(ses.mistake_counts, es.mistake_counts)
    if with_splits:
        assert ses.split_mistake_summary() == es.split_mistake_summary()
        assert all(" mistake_rate(%):" in l for l in ses.split_lines())
    else:
        assert int(ses.mistake_counts[0, 0]) == 2 * (steps * B - 1)
        assert ses.mistake_summary() == es.mistake_summary() or not torch.equal(ses.idx[0], es.idx[0])
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
        from hgrnet_b200.dist import MistakeShard, ShardedEvalStream, SplitShard
        from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
        h = synthetic_hierarchy(scaled_levels(21841), seed=1)
        u, x, targets = tss._case("hops", 512, 1024, 21841, 20842)
        tab = _table(h.c2p)
        ses = ShardedEvalStream(u.bank(), 0, batch=512, K=K, steps=4, splits=SplitShard(u, rank, world),
                                mistakes=MistakeShard(type("M", (), tab)(), rank, world))
        for s in range(4):
            ses.dev_feats[s].copy_(x.float())
            ses.dev_labels[s].copy_(targets)
        ses.run()
        torch.cuda.synchronize()
        _, idx = ops.score_topk_splits(ops.normalize_rows(x.float()), u.bank(), u.group_end, u.group_splits, u.S,
                                       col_id=u.col_id)
        one = ops.new_mistake_counts(dev, u.S)
        ops.hier_mistakes(idx, targets, counts=one, node_splits=u.node_splits, **tab)
        got = ses.split_mistake_summary()
        from hgrnet_b200.evaluate import mistake_summary
        assert got == [mistake_summary(c) for c in 4 * one]
        ses.close()
        out.put(("ok", rank, got))
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
