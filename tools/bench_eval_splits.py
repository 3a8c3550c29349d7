"""Head-side cost of evaluating three nested test splits through the graph-replayed evaluator, cfg-2 shape: one
multi-split ``EvalStream`` against one ``EvalStream`` per split.

B = 512 images per batch, D = 1,024, the 12-level 21,841-node synthetic hierarchy (bench.py's), every node a train class,
three nested test splits of 1,549 / 7,860 / 20,842 classes (the sizes of the official 2-hops / 3-hops / all sets), every
row with its own label drawn from the largest split, fp32 features already on the device (``host_io=False``: the
head-side cost, without the feature copy each pass would add).  Per batch:

* (a) one ``EvalStream`` over the largest split alone -- what one line costs today;
* (b) three ``EvalStream``s, one per split -- the head-side cost of today's three runs;
* (c) one ``EvalStream(splits=SplitEval)`` -- one pass, three lines.

Both without and with TOR / POR (``hier_metrics``).  The three variants are timed in alternating blocks of ``--steps``
batches, ``--reps`` times, in one process (CUDA events); the banks (43 MB at most) stay resident in the 126 MB L2, as in
a real evaluation loop.  A separate ``torch.profiler`` pass over eager multi-split calls reports the kernel times of the
scoring kernel and of the per-split merge.  Prints one JSON line with the median microseconds per batch, (c) / (a),
(c) / (b), the card's name and power limit; ``--out`` also writes it to a file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card_info():
    """Name and power limit of GPU 0 (a query only)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:                              # noqa: BLE001 -- the numbers stand without it, say so
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="batches per timed block")
    ap.add_argument("--reps", type=int, default=7, help="alternating blocks per variant")
    ap.add_argument("--out", default="")
    args = ap.parse_args(argv)

    import tempfile

    import numpy as np
    import torch

    from hgrnet_b200 import ops
    from hgrnet_b200.evaluate import HierMetrics, SplitEval
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    from hgrnet_b200.stream import EvalStream
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings

    if not torch.cuda.is_available():
        raise SystemExit("bench_eval_splits needs a CUDA device")
    dev = torch.device("cuda", 0)
    B, D, sizes, slots = 512, 1024, (1549, 7860, 20842), 8
    h = synthetic_hierarchy(scaled_levels(21841), seed=1)                 # bench.py's hierarchy
    N = len(h)
    nodes = np.random.default_rng(0).choice(N, size=sizes[-1], replace=False)
    split_ids = {"2-hops": nodes[:sizes[0]], "3-hops": nodes[:sizes[1]], "all": nodes}
    opts = parse_args([])
    opts.device = 0
    opts.folder = tempfile.mkdtemp()
    model = tree_model(opts, h.nodes, [h.nodes[i] for i in nodes], clip_model=TableEncoder(
        synthetic_embeddings(N, D, 1, normalize=False)).to(dev), hierarchy=h, node_tokens=node_id_tokens(N)).to(dev)
    model.update_classifier()
    g = torch.Generator().manual_seed(2)
    feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev) for i in range(slots)]
    labels = [torch.from_numpy(nodes[torch.randint(0, sizes[-1], (B,), generator=g).numpy()]).to(torch.int32).to(dev)
              for _ in range(slots)]

    def fill(es):
        for s in range(slots):
            es.dev_feats[s].copy_(feats[s])
            es.dev_labels[s].copy_(labels[s])
        return es

    def split_bank(ids):
        order = torch.from_numpy(np.sort(ids)).to(dev)
        return model.zsl_weights[order].contiguous(), order.to(torch.int32)

    result = {"card": card_info(), "B": B, "D": D, "split_sizes": list(sizes), "steps_per_block": args.steps,
              "reps": args.reps}
    for hier in (False, True):
        mk = lambda bank, cid: fill(EvalStream(bank, col_id=cid, batch=B, slots=slots, streams=2, host_io=False,
                                               hier=HierMetrics(model) if hier else None))
        per = [mk(*split_bank(split_ids[k])) for k in ("2-hops", "3-hops", "all")]
        multi = fill(EvalStream(model.bank_test, col_id=model._test_index_i32, batch=B, slots=slots, streams=2,
                                host_io=False, splits=SplitEval(model, split_ids, hier=hier)))
        variants = {"a_largest_split": [per[2]], "b_one_stream_per_split": per, "c_multi_split": [multi]}
        times = {k: [] for k in variants}
        for r in range(args.reps + 1):                   # block 0 warms up
            order = list(variants)[r % 3:] + list(variants)[:r % 3]
            for name in order:
                streams = variants[name]
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for es in streams:
                    es.begin()
                for i in range(args.steps):
                    for es in streams:
                        es.step(i % slots)
                for es in streams:
                    es.end()
                e1.record()
                e1.synchronize()
                if r > 0:
                    times[name].append(e0.elapsed_time(e1) * 1e3 / args.steps)
        med = {k: statistics.median(v) for k, v in times.items()}
        result["tor_por" if hier else "hits_only"] = {
            "us_per_batch_median": med, "us_per_batch_min": {k: min(v) for k, v in times.items()},
            "c_over_a": med["c_multi_split"] / med["a_largest_split"],
            "c_over_b": med["c_multi_split"] / med["b_one_stream_per_split"]}

    # kernel times of one eager multi-split call (no graph), in a run of its own
    se = SplitEval(model, split_ids, hier=False)
    x = ops.normalize_rows(feats[0])
    for _ in range(5):
        se.update(x, labels[0])
    torch.cuda.synchronize()
    result["multi_split_rescans_one_batch"] = ops.last_rescan_count()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(50):
            se.update(x, labels[i % slots])
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if "score_umma_pair_kernel" in ev.key or "topk_split_merge_kernel" in ev.key:
            name = "scoring_kernel" if "score_umma" in ev.key else "split_merge_kernel"
            kern[name] = {"us_mean": ev.device_time_total / max(ev.count, 1), "count": ev.count}
    result["kernels_eager_multi_split"] = kern
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
