"""Several test splits through the class-sharded evaluator (``ShardedEvalStream``), cfg-5 shape: one multi-split sharded
stream against one sharded stream per split.

Launch with ``python -m torch.distributed.run --nproc-per-node G tools/bench_splits_sharded.py`` (G = 1 runs as a plain
script too).  B = 4,096 images per batch, D = 1,024, the 12-level 21,841-node synthetic hierarchy (bench.py's), every
node a train class, three nested test splits of 1,549 / 7,860 / 20,842 classes (tools/bench_eval_splits.py's), every row
with its own label drawn from the largest split, features already on the device.  Per batch:

* (a) one sharded stream over the largest split alone -- what one line costs today;
* (b) three sharded streams, one per split -- today's three passes over the images;
* (c) one ``ShardedEvalStream(splits=SplitShard)`` -- one pass, three lines.

Each without and with TOR / POR.  The variants are timed in alternating blocks of ``--replays`` graph replays of
``--steps`` batches in one process (CUDA events around each block, ranks aligned by a barrier); the per-batch
microseconds of a block are the maximum over ranks and the medians are reported.  The banks (43 MB at most per rank)
stay resident in the 126 MB L2, as in a real evaluation loop.  A separate ``torch.profiler`` pass over eager (uncaptured)
multi-split batches gives the kernel times of the grouped scoring kernel, the producer-side split merge and the owner
merge, and the owner repair counter is reported.  Rank 0 prints one JSON line with the card's name and power limit;
``--out`` also writes it to a file.
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
    ap.add_argument("--steps", type=int, default=16, help="batches per captured graph")
    ap.add_argument("--replays", type=int, default=10, help="graph replays per timed block")
    ap.add_argument("--reps", type=int, default=7, help="timed blocks per variant (alternated)")
    ap.add_argument("--out", default=None, help="rank 0 also writes the JSON result to this file")
    args = ap.parse_args(argv)

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench_splits_sharded.py needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from hgrnet_b200.dist import HierShard, ShardedEvalStream, SplitShard, shard_bounds
    from hgrnet_b200.evaluate import HierMetrics, SplitEval
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings

    B, D, sizes = 4096, 1024, (1549, 7860, 20842)
    h = synthetic_hierarchy(scaled_levels(21841), seed=1)                 # bench.py's hierarchy
    N = len(h)
    nodes = np.random.default_rng(0).choice(N, size=sizes[-1], replace=False)
    split_ids = {"2-hops": nodes[:sizes[0]], "3-hops": nodes[:sizes[1]], "all": nodes}
    opts = parse_args([])
    opts.device = local
    opts.folder = tempfile.mkdtemp()
    model = tree_model(opts, h.nodes, [h.nodes[i] for i in nodes], clip_model=TableEncoder(
        synthetic_embeddings(N, D, 1, normalize=False)).to(dev), hierarchy=h, node_tokens=node_id_tokens(N)).to(dev)
    model.eval()
    model.update_classifier()
    g = torch.Generator().manual_seed(2)
    feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev) for i in range(8)]
    labels = [torch.from_numpy(nodes[torch.randint(0, sizes[-1], (B,), generator=g).numpy()]).to(torch.int32).to(dev)
              for _ in range(8)]

    def fill(ses):
        for s in range(args.steps):
            ses.dev_feats[s].copy_(feats[s % 8])
            ses.dev_labels[s].copy_(labels[s % 8])
        return ses

    def split_stream(ids, hier):
        """A plain sharded stream over one split: its classes in node order, rows shard_bounds-cut."""
        order = torch.from_numpy(np.sort(ids)).to(dev)
        lo, hi = shard_bounds(len(ids), world)[rank]
        bank = model.zsl_weights[order[lo:hi]].contiguous()
        return fill(ShardedEvalStream(bank, lo, batch=B, steps=args.steps, col_id=order[lo:hi].to(torch.int32),
                                      hier=hier))

    def block(streams):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.replays):
            for ses in streams:
                ses.run()
        e1.record()
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e3 / (args.replays * args.steps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    result = {"card": card_info(), "G": world, "B": B, "D": D, "split_sizes": list(sizes), "steps_per_graph": args.steps,
              "replays_per_block": args.replays, "reps": args.reps,
              "inputs": "device-resident fp32 features (8 batches rotated), banks resident in L2",
              "timing": "CUDA events per block of replays, max over ranks, median over blocks"}
    for hier in (False, True):
        hs = HierShard(HierMetrics(model).rows_args(), rank, world) if hier else None
        per = [split_stream(split_ids[k], hs) for k in ("2-hops", "3-hops", "all")]
        se = SplitEval(model, split_ids, hier=hier)
        sh = SplitShard(se, rank, world)
        multi = fill(ShardedEvalStream(se.bank(), 0, batch=B, steps=args.steps, splits=sh))
        variants = {"a_largest_split": [per[2]], "b_one_stream_per_split": per, "c_multi_split": [multi]}
        times = {k: [] for k in variants}
        for r in range(args.reps + 1):                   # block 0 warms up
            order = list(variants)[r % 3:] + list(variants)[:r % 3]
            for name in order:
                t = block(variants[name])
                if r > 0:
                    times[name].append(t)
        med = {k: statistics.median(v) for k, v in times.items()}
        lines = multi.split_lines()
        key = "tor_por" if hier else "hits_only"
        result[key] = {"us_per_batch_median": med, "us_per_batch_blocks": times,
                       "c_over_a": med["c_multi_split"] / med["a_largest_split"],
                       "c_over_b": med["c_multi_split"] / med["b_one_stream_per_split"],
                       "owner_repairs": int(multi.repairs.item()), "lines": lines,
                       "rank0_local_group_end": sh.group_end}
        if rank == 0:
            print("G = %d %s: (a) %.2f  (b) %.2f  (c) %.2f us/batch  c/a %.3f  c/b %.3f  repairs %d" % (
                world, key, med["a_largest_split"], med["b_one_stream_per_split"], med["c_multi_split"],
                result[key]["c_over_a"], result[key]["c_over_b"], result[key]["owner_repairs"]), flush=True)
        for ses in per + [multi]:
            ses.close()
        del per, multi

    # kernel times of eager multi-split batches (no graph), in a run of its own
    se = SplitEval(model, split_ids, hier=False)
    ses = fill(ShardedEvalStream(se.bank(), 0, batch=B, steps=args.steps, splits=SplitShard(se, rank, world),
                                 use_graph=False))
    for _ in range(3):
        ses.run()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            ses.run()
        torch.cuda.synchronize()
    kern = {}
    names = {"score_umma_pair_kernel": "grouped_scoring_kernel", "topk_split_merge_kernel": "producer_split_merge",
             "topk_split_cert_kernel": "owner_split_merge"}
    for ev in prof.key_averages():
        for pat, name in names.items():
            if pat in ev.key:
                kern[name] = {"us_mean": ev.device_time_total / max(ev.count, 1), "count": ev.count}
    t = torch.tensor([kern.get(n, {}).get("us_mean", 0.0) for n in names.values()], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    result["kernels_eager_multi_split_us_max_over_ranks"] = dict(zip(names.values(), t.tolist()))
    result["kernels_eager_multi_split_rank0"] = kern
    result["owner_repairs_eager"] = int(ses.repairs.item())
    ses.close()
    if rank == 0:
        line = json.dumps(result)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
