"""Cost of TOR / POR inside the class-sharded evaluator (``ShardedEvalStream`` with ``hier``), cfg-5 shape.

Launch with ``python -m torch.distributed.run --nproc-per-node G tools/bench_hier_sharded.py`` (G = 1 runs as a plain
script too).  B = 4,096 images per batch, C = 21,841 classes (every node a test class), D = 1,024, the 12-level synthetic
hierarchy; every rank holds 1/G of the class bank and 1/G of the level-sorted train bank.  Two train splits:

* ``all``:  every node is a train class (M = 21,841 train columns, 2,731 per rank at G = 8);
* ``real``: 1,000 leaves plus their ancestors (``tools/bench_hier_stream.real_split``).

Inputs are device-resident: several copies of the rank's class-bank shard and 8 feature batches, rotated so that the
operands of one graph replay exceed the 126 MB L2 (the train-bank slice is one tensor, as in real use).  For each split
the stream with metrics off and the stream with metrics on are timed in alternating blocks of ``--replays`` graph
replays in one process (CUDA events around each block, ranks aligned by a barrier); the per-batch microseconds of a
block are the maximum over ranks, and the medians are printed with the card's name and power limit.  ``--dry-run``
prints the shape arithmetic only and needs no GPU.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_hier_stream import L2_BYTES, card_info, real_split  # noqa: E402


def shapes(B: int, C: int, D: int, M: int, n_levels: int, G: int, steps: int):
    """Per-rank bytes and operations of one batch at G ranks; bank copies the rotation needs to exceed L2."""
    shard_c = -(-C // G)
    shard_m = -(-M // G)
    shard_bytes = shard_c * D * 2
    n_bank = min(steps, max(2, math.ceil(1.6 * L2_BYTES / shard_bytes)))
    return {"G": G, "B": B, "C": C, "D": D, "train_cols": M, "class_cols_per_rank": shard_c,
            "train_cols_per_rank": shard_m, "n_bank": n_bank, "n_feat": 8,
            "rotated_bytes_per_replay": n_bank * shard_bytes + 8 * B * D * 2,
            "score_gflop_per_rank": 2.0 * B * shard_c * D / 1e9, "hier_gflop_per_rank": 2.0 * B * shard_m * D / 1e9,
            "hier_words_pushed_bytes_per_rank": B * n_levels * 8}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--classes", type=int, default=21841)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=16, help="batches per captured graph")
    ap.add_argument("--replays", type=int, default=10, help="graph replays per timed block")
    ap.add_argument("--reps", type=int, default=9, help="timed blocks per configuration (alternated)")
    ap.add_argument("--split", choices=("all", "real", "both"), default="both")
    ap.add_argument("--gpus", type=int, default=None, help="with --dry-run: the G to do the arithmetic for")
    ap.add_argument("--out", default=None, help="rank 0 also writes the JSON result to this file")
    ap.add_argument("--dry-run", action="store_true", help="print the shape arithmetic only (no GPU)")
    args = ap.parse_args(argv)

    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    B, C, D = args.batch, args.classes, args.dim
    h = synthetic_hierarchy(scaled_levels(C), seed=1)                   # bench.py's hierarchy
    n_levels = h.max_depth + 1
    splits = {"all": list(range(C)), "real": real_split(h)}
    names = ["all", "real"] if args.split == "both" else [args.split]
    if args.dry_run:
        Gs = [args.gpus] if args.gpus else [1, 2, 4, 8]
        print(json.dumps({"dry_run": True, "levels": n_levels,
                          "shapes": {n: [shapes(B, C, D, len(splits[n]), n_levels, G, args.steps) for G in Gs]
                                     for n in names}}))
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench_hier_sharded.py needs a CUDA device (use --dry-run for the shape arithmetic)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from hgrnet_b200.dist import HierShard, ShardedEvalStream, shard_bounds
    from hgrnet_b200.evaluate import HierMetrics
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings
    table = synthetic_embeddings(C, D, 1, normalize=False)
    g = torch.Generator().manual_seed(7)
    feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev).to(torch.bfloat16) for i in range(8)]
    labels = [torch.randint(0, C, (B,), generator=g, dtype=torch.int32).to(dev) for _ in range(8)]
    result = {"card": card_info(), "G": world, "B": B, "C": C, "D": D, "levels": n_levels, "steps_per_graph": args.steps,
              "replays_per_block": args.replays, "reps": args.reps,
              "inputs": "device-resident bf16, class-bank shard copies and 8 feature batches rotated past L2",
              "timing": "CUDA events per block of replays, max over ranks, median over blocks", "splits": {}}
    lo, hi = shard_bounds(C, world)[rank]

    def block(ses):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.replays):
            ses.run()
        e1.record()
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e3 / (args.replays * args.steps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for name in names:
        p = shapes(B, C, D, len(splits[name]), n_levels, world, args.steps)
        opts = parse_args([])
        opts.device, opts.folder, opts.weights = local, "/tmp/hgr_bench_hier_sharded_out", "equal"
        model = tree_model(opts, [h.nodes[i] for i in splits[name]], h.nodes, clip_model=TableEncoder(table).to(dev),
                           hierarchy=h, node_tokens=node_id_tokens(C))
        model.eval()
        model.update_classifier()
        ids = model._test_index_i32[lo:hi].contiguous()
        banks = [model.bank_test[lo:hi].clone() for _ in range(p["n_bank"])]
        hier = HierShard(HierMetrics(model).rows_args(), rank, world)
        streams = {}
        for mode in ("off", "on"):
            ses = ShardedEvalStream(banks[0], lo, batch=B, steps=args.steps, banks=banks, col_id=ids,
                                    feat_dtype=torch.bfloat16, hier=hier if mode == "on" else None)
            for s in range(args.steps):
                ses.dev_feats[s].copy_(feats[s % 8])
                ses.dev_labels[s].copy_(labels[s % 8])
            streams[mode] = ses
        for ses in streams.values():
            block(ses)                                                  # warm-up
        times = {"off": [], "on": []}
        for _ in range(args.reps):
            for mode in ("off", "on"):
                times[mode].append(block(streams[mode]))
        med = {m: sorted(t)[len(t) // 2] for m, t in times.items()}
        hits_off, hits_on = streams["off"].all_reduce_hits().tolist(), streams["on"].all_reduce_hits().tolist()
        assert hits_off == hits_on, (hits_off, hits_on)                 # the same batches were scored
        ratios = streams["on"].hier_ratios()
        result["splits"][name] = {**p, "us_per_batch_off": med["off"], "us_per_batch_on": med["on"],
                                  "added_us": med["on"] - med["off"], "ratio": med["on"] / med["off"],
                                  "blocks_us_off": times["off"], "blocks_us_on": times["on"], "hier_ratios": ratios}
        if rank == 0:
            print("G = %d %-4s M = %5d (%d per rank): metrics off %.2f us/batch, on %.2f us/batch (+%.2f us, %.3fx)"
                  % (world, name, p["train_cols"], p["train_cols_per_rank"], med["off"], med["on"],
                     med["on"] - med["off"], med["on"] / med["off"]), flush=True)
        for ses in streams.values():
            ses.close()
        del streams, banks, model, hier
        torch.cuda.synchronize()
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
