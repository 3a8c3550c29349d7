"""Cost of the per-class Hit@k table (``hgr_class_hits``, class-averaged Hit@k) in the evaluators.

Workloads, on the 21,841-node synthetic hierarchy (bench.py's), test classes = 20,842 of its nodes, fp32 features
already on the device:

* cfg 2: ``EvalStream`` (one GPU, graph-replayed), B = 512, D = 1,024, hits only -- without and with ``classes``; once
  with a random label per row, once with one label per batch (the reference's class-grouped test loader: every row of
  a batch adds to the same six counters, the kernel's contention case);
* cfg 5: ``ShardedEvalStream(splits=...)`` at G = 1, B = 4,096, D = 1,024, the three nested test splits of 1,549 /
  7,860 / 20,842 classes (tools/bench_splits_sharded.py's), per-row labels -- without and with ``classes`` (one table
  per split).

The two variants of a workload are timed in alternating blocks (CUDA events around each block) and the medians are
reported.  The banks stay resident in the 126 MB L2, as in a real evaluation loop.  The kernel alone is timed with CUDA
events over many eager launches on the lists the streams produced.  Prints one JSON line with the card's name and power
limit; ``--out`` also writes it to a file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_eval_splits import card_info  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="cfg 2: batches per timed block")
    ap.add_argument("--sharded_steps", type=int, default=16, help="cfg 5: batches per captured graph")
    ap.add_argument("--replays", type=int, default=10, help="cfg 5: graph replays per timed block")
    ap.add_argument("--reps", type=int, default=9, help="alternating timed blocks per variant")
    ap.add_argument("--kernel_iters", type=int, default=2000, help="eager launches per kernel timing")
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_class_hits.py needs a CUDA device")
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import ShardedEvalStream, SplitShard
    from hgrnet_b200.evaluate import ClassHits, SplitEval
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    from hgrnet_b200.stream import EvalStream
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings

    dev = torch.device("cuda", 0)
    D, sizes, slots = 1024, (1549, 7860, 20842), 8
    h = synthetic_hierarchy(scaled_levels(21841), seed=1)
    N = len(h)
    nodes = np.random.default_rng(0).choice(N, size=sizes[-1], replace=False)
    split_ids = {"2-hops": nodes[:sizes[0]], "3-hops": nodes[:sizes[1]], "all": nodes}
    opts = parse_args([])
    opts.device = 0
    opts.folder = tempfile.mkdtemp()
    model = tree_model(opts, h.nodes, [h.nodes[i] for i in nodes], clip_model=TableEncoder(
        synthetic_embeddings(N, D, 1, normalize=False)).to(dev), hierarchy=h, node_tokens=node_id_tokens(N)).to(dev)
    model.eval()
    model.update_classifier()
    ch = ClassHits(model)

    def batches(B, single_label):
        g = torch.Generator().manual_seed(2)
        feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev) for i in range(slots)]
        if single_label:
            pick = torch.randint(0, sizes[-1], (slots,), generator=g).numpy()
            labels = [torch.full((B,), int(nodes[pick[i]]), dtype=torch.int32, device=dev) for i in range(slots)]
        else:
            labels = [torch.from_numpy(nodes[torch.randint(0, sizes[-1], (B,), generator=g).numpy()]).to(torch.int32)
                      .to(dev) for _ in range(slots)]
        return feats, labels

    def alternate(variants, block):
        times = {k: [] for k in variants}
        for r in range(args.reps + 1):                   # block 0 warms up
            order = list(variants)[r % 2:] + list(variants)[:r % 2]
            for name in order:
                t = block(variants[name])
                if r > 0:
                    times[name].append(t)
        med = {k: statistics.median(v) for k, v in times.items()}
        return {"us_per_batch_median": med, "us_per_batch_blocks": times,
                "overhead_us_per_batch": med["with_classes"] - med["without"]}

    def kernel_us(idx, targets, node_splits, n_sets):
        counts = ops.new_class_counts(dev, N, n_sets)
        for _ in range(20):
            ops.class_hits(idx, targets, counts, node_splits=node_splits)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.kernel_iters):
            ops.class_hits(idx, targets, counts, node_splits=node_splits)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / args.kernel_iters

    def kernel_us_graph(idx, targets, node_splits, n_sets, launches=100, replays=20):
        """The same launches captured in one CUDA graph: the device time per launch without the host's launch gaps."""
        counts = ops.new_class_counts(dev, N, n_sets)
        st = torch.cuda.Stream(device=dev)
        st.wait_stream(torch.cuda.current_stream(dev))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(st):
            ops.class_hits(idx, targets, counts, node_splits=node_splits)
            st.synchronize()
            with torch.cuda.graph(g, stream=st):
                for _ in range(launches):
                    ops.class_hits(idx, targets, counts, node_splits=node_splits)
        torch.cuda.synchronize(dev)
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(replays):
            g.replay()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (replays * launches)

    result = {"card": card_info(), "D": D, "n_nodes": N, "test_classes": sizes[-1], "split_sizes": list(sizes),
              "reps": args.reps, "inputs": "device-resident fp32 features, banks resident in L2",
              "timing": "CUDA events per block, variants alternated, median over blocks; kernel_us: CUDA events over "
                        "eager launches (includes the host's launch gaps of back-to-back launches); kernel_us_graph: "
                        "CUDA events over replays of one graph of 100 launches"}

    # ---- cfg 2: EvalStream, B = 512 -------------------------------------------------------------------------------
    B = 512
    variants = {k: [EvalStream(model.bank_test, col_id=model._test_index_i32, batch=B, slots=slots, streams=2,
                               host_io=False, classes=c)] for k, c in (("without", None), ("with_classes", ch))}

    def block(streams):
        es = streams[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        es.begin()
        for i in range(args.steps):
            es.step(i % slots)
        es.end()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / args.steps

    for name, single in (("cfg2_eval_stream_row_labels", False), ("cfg2_eval_stream_one_label_per_batch", True)):
        feats, labels = batches(B, single)
        for v in variants.values():
            es = v[0]
            for s in range(slots):
                es.dev_feats[s].copy_(feats[s])
                es.dev_labels[s].copy_(labels[s])
            es.tally.zero_()                             # the summary covers this workload only
        cfg2 = alternate(variants, block)
        es = variants["with_classes"][0]
        cfg2["kernel_us"] = kernel_us(es.idx[0], es.dev_labels[0], None, 1)
        cfg2["kernel_us_graph"] = kernel_us_graph(es.idx[0], es.dev_labels[0], None, 1)
        cfg2["summary"] = es.class_summary()
        cfg2["B"] = B
        result[name] = cfg2
        print("%s: without %.2f  with %.2f us/batch  kernel %.2f us eager, %.2f us in a graph" % (
            name, cfg2["us_per_batch_median"]["without"], cfg2["us_per_batch_median"]["with_classes"],
            cfg2["kernel_us"], cfg2["kernel_us_graph"]), flush=True)
    del variants, es

    # ---- cfg 5: ShardedEvalStream(splits=...), G = 1, B = 4,096 --------------------------------------------------
    B = 4096
    feats, labels = batches(B, False)
    se = SplitEval(model, split_ids, hier=False)
    sh = SplitShard(se, 0, 1)

    def sfill(ses):
        for s in range(args.sharded_steps):
            ses.dev_feats[s].copy_(feats[s % slots])
            ses.dev_labels[s].copy_(labels[s % slots])
        return ses

    variants = {k: [sfill(ShardedEvalStream(se.bank(), 0, batch=B, steps=args.sharded_steps, splits=sh, classes=c))]
                for k, c in (("without", None), ("with_classes", ch))}

    def sblock(streams):
        ses = streams[0]
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.replays):
            ses.run()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (args.replays * args.sharded_steps)

    cfg5 = alternate(variants, sblock)
    ses = variants["with_classes"][0]
    cfg5["kernel_us"] = kernel_us(ses.idx[0], ses.dev_labels[0], sh.node_splits, sh.S)
    cfg5["kernel_us_graph"] = kernel_us_graph(ses.idx[0], ses.dev_labels[0], sh.node_splits, sh.S)
    cfg5["split_summary"] = ses.split_class_summary()
    cfg5["owner_repairs"] = int(ses.repairs.item())
    cfg5["B"], cfg5["G"], cfg5["steps_per_graph"], cfg5["replays_per_block"] = B, 1, args.sharded_steps, args.replays
    result["cfg5_sharded_splits_G1"] = cfg5
    print("cfg 5 ShardedEvalStream(splits) G = 1: without %.2f  with %.2f us/batch  kernel %.2f us eager, %.2f us in a "
          "graph" % (cfg5["us_per_batch_median"]["without"], cfg5["us_per_batch_median"]["with_classes"],
                     cfg5["kernel_us"], cfg5["kernel_us_graph"]), flush=True)
    for v in variants.values():
        v[0].close()

    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
