"""Cost of TOR / POR inside the graph-replayed evaluator (``EvalStream`` with ``hier``), cfg-2 shape.

B = 512 images per batch, C = 21,841 classes (every node a test class), D = 1,024, the 12-level synthetic hierarchy.
Inputs are device-resident and rotated as in bench.py: several copies of the test-class bank, together larger than
the 126 MB L2, and 8 feature batches; every row has its own random label.  The level-sorted train bank is one tensor,
as in real use.  Two train splits:

* ``all``:  every node is a train class (M = 21,841 train columns);
* ``real``: 1,000 leaves plus their ancestors, the shape of the reference's ImageNet-21K split.

For each split the stream with metrics off and the stream with metrics on are timed in alternating blocks of
``--steps`` batches in one process (CUDA events around each block); the median per-batch microseconds are printed with
the card's name and power limit.  ``--dry-run`` prints the shape arithmetic only and needs no GPU.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

L2_BYTES = 126e6


def real_split(h, n_leaves: int = 1000, seed: int = 0):
    """Node ids of ``n_leaves`` leaves (seeded draw) plus all their ancestors, ascending."""
    import numpy as np
    leaves = [n for n in range(len(h)) if not h.p2c[n]]
    pick = np.random.RandomState(seed).choice(len(leaves), size=min(n_leaves, len(leaves)), replace=False)
    chosen = {leaves[i] for i in pick}
    return sorted(chosen | {p for n in chosen for p in h.c2p[n]})


def shapes(B: int, C: int, D: int, train_cols: int):
    """Bytes and operations of one batch; how many bank copies the rotation needs to exceed L2 (as bench.py)."""
    bank_bytes = C * D * 2
    n_bank = max(2, math.ceil(1.6 * L2_BYTES / bank_bytes))
    n_feat = 8
    return {"B": B, "C": C, "D": D, "train_cols": train_cols, "bank_bytes": bank_bytes, "n_bank": n_bank,
            "n_feat": n_feat, "slots": n_bank * n_feat // math.gcd(n_bank, n_feat),
            "rotated_bytes": n_bank * bank_bytes + n_feat * B * D * 2,
            "train_bank_bytes": train_cols * D * 2,
            "score_gflop": 2.0 * B * C * D / 1e9, "hier_gflop": 2.0 * B * train_cols * D / 1e9}


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
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--classes", type=int, default=21841)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=400, help="batches per timed block")
    ap.add_argument("--reps", type=int, default=11, help="timed blocks per configuration (alternated)")
    ap.add_argument("--streams", type=int, default=6, help="streams the slots' graphs are replayed on (bench.py's default)")
    ap.add_argument("--split", choices=("all", "real", "both"), default="both")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    ap.add_argument("--dry-run", action="store_true", help="print the shape arithmetic only (no GPU)")
    args = ap.parse_args(argv)

    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    B, C, D = args.batch, args.classes, args.dim
    h = synthetic_hierarchy(scaled_levels(C), seed=1)                   # bench.py's hierarchy
    splits = {"all": list(range(C)), "real": real_split(h)}
    names = ["all", "real"] if args.split == "both" else [args.split]
    plan = {n: shapes(B, C, D, len(splits[n])) for n in names}
    if args.dry_run:
        print(json.dumps({"dry_run": True, "levels": h.max_depth + 1, "shapes": plan}))
        return 0

    import torch
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings
    if not torch.cuda.is_available():
        raise SystemExit("bench_hier_stream.py needs a CUDA device (use --dry-run for the shape arithmetic)")
    dev = torch.device("cuda", 0)
    table = synthetic_embeddings(C, D, 1, normalize=False)
    g = torch.Generator().manual_seed(7)
    result = {"card": card_info(), "B": B, "C": C, "D": D, "steps_per_block": args.steps, "reps": args.reps,
              "streams": args.streams, "inputs": "device-resident bf16, test banks rotated over more bytes than L2",
              "splits": {}}
    for name in names:
        p = plan[name]
        opts = parse_args([])
        opts.device, opts.folder, opts.weights = 0, "/tmp/hgr_bench_hier_out", "equal"
        model = tree_model(opts, [h.nodes[i] for i in splits[name]], h.nodes, clip_model=TableEncoder(table).to(dev),
                           hierarchy=h, node_tokens=node_id_tokens(C))
        model.eval()
        model.update_classifier()
        banks = [model.bank_test.clone() for _ in range(p["n_bank"])]
        feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev).to(torch.bfloat16) for i in range(p["n_feat"])]
        labels = [torch.randint(0, C, (B,), generator=g, dtype=torch.int32).to(dev) for _ in range(p["n_feat"])]
        streams = {}
        for mode in ("off", "on"):
            es = model.make_eval_stream(batch=B, slots=p["slots"], streams=args.streams, banks=banks, host_io=False,
                                        feat_dtype=torch.bfloat16, hier_metrics=mode == "on")
            for s in range(p["slots"]):
                es.dev_feats[s].copy_(feats[s % p["n_feat"]])
                es.dev_labels[s].copy_(labels[s % p["n_feat"]])
            streams[mode] = es

        def block(es):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            es.begin()
            for i in range(args.steps):
                es.step(i % p["slots"])
            es.end()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) * 1e3 / args.steps

        for es in streams.values():
            block(es)                                                   # warm-up
        times = {"off": [], "on": []}
        for _ in range(args.reps):
            for mode in ("off", "on"):
                times[mode].append(block(streams[mode]))
        med = {m: sorted(t)[len(t) // 2] for m, t in times.items()}
        hits_off, hits_on = streams["off"].hit_counts(), streams["on"].hit_counts()
        assert hits_off == hits_on, (hits_off, hits_on)                 # the same batches were scored
        result["splits"][name] = {"train_cols": p["train_cols"], "us_per_batch_off": med["off"],
                                  "us_per_batch_on": med["on"], "added_us": med["on"] - med["off"],
                                  "ratio": med["on"] / med["off"], "blocks_us_off": times["off"],
                                  "blocks_us_on": times["on"], "hier_ratios": streams["on"].hier_ratios()}
        print("%-4s M = %5d: metrics off %.2f us/batch, on %.2f us/batch (+%.2f us, %.2fx)"
              % (name, p["train_cols"], med["off"], med["on"], med["on"] - med["off"], med["on"] / med["off"]))
        del streams, banks, model
        torch.cuda.synchronize()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
