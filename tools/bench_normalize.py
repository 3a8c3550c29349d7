"""Time the row normalise (``normalize_rows_kernel``) at the shapes it runs at, through ``ops.normalize_rows_dual``
(the same kernel as ``ops.normalize_rows``, writing into a given bf16 buffer).

    python tools/bench_normalize.py [--reps 200]

(a) the streaming evaluator's per-batch normalise: B = 512 bf16 feature rows of D = 1,024 into bf16, launched
back to back inside one CUDA graph (the batch stays in L2, as it does in the evaluator); (b) the class-bank build:
21,841 rows of D = 1,024 from fp32 and from bf16 into bf16, two input copies alternated so that the 134 MB / 89 MB
working set does not sit in L2.  Prints one JSON line: microseconds per launch, and for (b) the bytes moved per
microsecond.  HGR_LIB selects a library variant, as for every tool here.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200, help="launches per graph")
    ap.add_argument("--graphs", type=int, default=7, help="graph replays timed (median reported)")
    args = ap.parse_args()

    import torch
    from hgrnet_b200 import ops

    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)

    def time_us(fn, n_inputs):
        for i in range(n_inputs):   # warm-up, lazy module loading
            fn(i)
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(st), torch.cuda.graph(graph, stream=st):
            for i in range(args.reps):
                fn(i % n_inputs)
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.graphs):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            graph.replay()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) * 1e3 / args.reps)
        times.sort()
        return times[len(times) // 2]

    out = {"gpu": torch.cuda.get_device_name(dev), "reps_per_graph": args.reps, "graphs": args.graphs}
    x = torch.randn(512, 1024, device=dev, generator=g).to(torch.bfloat16)
    o = torch.empty(512, 1024, device=dev, dtype=torch.bfloat16)
    out["batch_512_bf16_us"] = time_us(lambda i: ops.normalize_rows_dual(x, o), 1)
    C, D = 21841, 1024
    for dt, name in ((torch.float32, "bank_fp32"), (torch.bfloat16, "bank_bf16")):
        ins = [torch.randn(C, D, device=dev, generator=g).to(dt) for _ in range(2)]
        outs = [torch.empty(C, D, device=dev, dtype=torch.bfloat16) for _ in range(2)]
        us = time_us(lambda i: ops.normalize_rows_dual(ins[i], outs[i]), 2)
        moved = C * D * (ins[0].element_size() + 2)
        out[name + "_us"] = us
        out[name + "_GBps"] = moved / us / 1e3
    print(json.dumps(out))


if __name__ == "__main__":
    main()
