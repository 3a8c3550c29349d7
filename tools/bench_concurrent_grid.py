"""Grid share sweep of the streaming evaluator (``EvalStream(concurrent=c)``, ``ops.score_topk(grid_share=c)``).

    python tools/bench_concurrent_grid.py [--shares 1,2,3,4] [--workloads cfg2,cfg5] [--reps 15] [--out FILE]

Per workload (bench.py's cfg 2: B = 512 and cfg 5: B = 4,096, both against 21,841 classes at D = 1,024, top-20):

* ``EvalStream`` on 6 round-robin streams, device-resident bf16 features, as bench.py's ``value``: the banks and feature
  batches rotate over more than 1.6 x the 126 MB L2 (one graph per (bank, batch) pair).  One ``EvalStream`` per share;
  blocks of ``--steps`` steps are timed with CUDA events, the shares alternating block by block, ``--reps`` rounds; the
  median block decides.
* the scoring kernel alone at every share (``HGR_IMPL_FLAG_NO_MERGE``), and the scoring call with its merge, one launch
  after another on one stream in one CUDA graph over the same rotated inputs: the merge is their difference.

Prints and writes one JSON object with the card's name, power limit and the SM clocks sampled while the blocks ran.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS, ClockSampler, _n_bank  # noqa: E402
from hgrnet_b200 import _cabi, ops  # noqa: E402
from hgrnet_b200.stream import EvalStream  # noqa: E402
from hgrnet_b200.synthetic import synthetic_embeddings  # noqa: E402

K = 20
N_FEAT = 8


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:   # the timing does not depend on it; report what failed
        return {"name": torch.cuda.get_device_name(0), "error": str(e)}


def graph_us(fn, n, min_ms=40.0):
    """`n` back-to-back calls fn(i) in one CUDA graph on a side stream, replayed for >= min_ms: us per call."""
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn(0)
        st.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for i in range(n):
                fn(i)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        g.replay()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    reps = int(max(3, min_ms / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (reps * n) * 1e3


def sweep(wl_key, shares, args, dev):
    wl = WORKLOADS[wl_key]
    B, C, D = wl["B"], wl["C"], wl["D"]
    bank0 = ops.normalize_rows(synthetic_embeddings(C, D, 1, normalize=False).to(dev).to(torch.bfloat16))
    n_bank = _n_bank(wl, 1)
    banks = [bank0] + [bank0.clone() for _ in range(n_bank - 1)]
    feats = [synthetic_embeddings(B, D, 100 + i, normalize=False).to(dev).to(torch.bfloat16) for i in range(N_FEAT)]
    g = torch.Generator().manual_seed(7)
    labels = [torch.full((B,), int(torch.randint(0, C, (1,), generator=g)), dtype=torch.int32, device=dev)
              for _ in range(N_FEAT)]
    slots = n_bank * N_FEAT // math.gcd(n_bank, N_FEAT)
    streams = {}
    for c in shares:
        es = EvalStream(bank0, batch=B, K=K, slots=slots, streams=args.streams, banks=banks, host_io=False,
                        feat_dtype=torch.bfloat16, concurrent=c)
        for s in range(slots):
            es.dev_feats[s].copy_(feats[s % N_FEAT])
            es.dev_labels[s].copy_(labels[s % N_FEAT])
        streams[c] = es

    def block(es):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        es.begin()
        for i in range(args.steps):
            es.step(i % slots)
        es.end()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / args.steps

    for es in streams.values():   # warm-up
        block(es)
    times = {c: [] for c in shares}
    sampler = ClockSampler(0)
    sampler.start()
    for r in range(args.reps):
        order = shares if r % 2 == 0 else shares[::-1]
        for c in order:
            times[c].append(block(streams[c]))
    clocks = sampler.stop()
    hits = {c: streams[c].hit_counts() for c in shares}
    plans = {c: streams[c].plan() for c in shares}
    del streams
    xs = [ops.normalize_rows(f) for f in feats]
    nm = ops.HGR_IMPL_TCGEN05 | _cabi.HGR_IMPL_FLAG_NO_MERGE
    out = {"B": B, "C": C, "D": D, "K": K, "streams": args.streams, "slots": slots, "banks": n_bank,
           "steps_per_block": args.steps, "blocks_per_share": args.reps,
           "policy_share": ops.score_topk_grid_share(B, C, D, K), "clocks": clocks, "shares": {}}
    for c in shares:
        ts = sorted(times[c])
        kern = graph_us(lambda i: ops.score_topk(xs[i % N_FEAT], banks[i % n_bank], K=K, impl=nm, grid_share=c), slots)
        call = graph_us(lambda i: ops.score_topk(xs[i % N_FEAT], banks[i % n_bank], targets=labels[i % N_FEAT], K=K,
                                                 impl=ops.HGR_IMPL_TCGEN05, grid_share=c), slots)
        out["shares"][str(c)] = {
            "plan": plans[c], "us_per_step_median": ts[len(ts) // 2], "us_per_step_min": ts[0],
            "us_per_step_max": ts[-1], "images_per_s_median": B / (ts[len(ts) // 2] * 1e-6),
            "kernel_alone_us": kern, "call_with_merge_us": call, "merge_us": call - kern,
            "hits_per_step": [h / (len(times[c]) + 1) / args.steps for h in hits[c]]}
        print("%s c=%d  %7.2f us/step (%.2f M images/s; min %.2f max %.2f)  kernel %.2f us  merge %.2f us  plan %s" % (
            wl_key, c, ts[len(ts) // 2], B / ts[len(ts) // 2], ts[0], ts[-1], kern, call - kern, plans[c]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shares", default="1,2,3,4")
    ap.add_argument("--workloads", default="cfg2,cfg5")
    ap.add_argument("--streams", type=int, default=6)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_concurrent_grid.py measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    shares = [int(c) for c in args.shares.split(",")]
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "workloads": {}}
    print("card: %s" % res["card"], flush=True)
    for wl in args.workloads.split(","):
        res["workloads"][wl] = sweep(wl, shares, args, dev)
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
