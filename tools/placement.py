"""Which SMs the small kernels of the streaming evaluator share with a scoring CTA (diagnostics build).

    tools/build_variant.sh placement -DHGR_PLACEMENT "score_pair.cu aggregate_norm.cu topk_merge.cu"
    python tools/placement.py [--steps 600] [--streams 6] [--out FILE]

Runs cfg 2 (B = 512, C = 21,841, D = 1,024, top-20) through ``EvalStream`` with device-resident bf16 features on the
library variant ``hgrnet_b200/lib/var_placement.so`` (HGR_LIB overrides), whose scoring, row-normalise and select-merge
kernels log per CTA the SM and %globaltimer at entry and exit (csrc/placement.cuh).  Reports, for the normalise and the
merge CTAs, the share of their CTA time during which a scoring CTA ran on the same SM, and the share of CTAs that saw
one at all; and the share of the top-K epilogue's chunks that found the candidate queue too full for the roomy append.
The instrumented kernels use more registers than the production ones (``footprint`` in the report is the variant's),
and %globaltimer ticks in steps of ``timer_step_ns``: read the shares with both in mind.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("HGR_LIB", os.path.join(ROOT, "hgrnet_b200", "lib", "var_placement.so"))

REC = np.dtype([("t0", "<u8"), ("t1", "<u8"), ("sm", "<u4"), ("kind", "<u4")])   # place::Rec
KINDS = {1: "score", 2: "normalize", 3: "merge"}


def overlap_report(rec: np.ndarray) -> dict:
    """Per small-kernel kind: CTA time overlapped by scoring CTAs on the same SM, over the total CTA time."""
    score = rec[rec["kind"] == 1]
    by_sm = {}
    for sm in np.unique(score["sm"]):
        s = score[score["sm"] == sm]
        order = np.argsort(s["t0"])
        merged = []   # union of the SM's scoring intervals
        for t0, t1 in zip(s["t0"][order].astype(np.int64), s["t1"][order].astype(np.int64)):
            if merged and t0 <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], t1)
            else:
                merged.append([t0, t1])
        by_sm[int(sm)] = np.array(merged, dtype=np.int64).reshape(-1, 2)
    out = {"score_ctas": int(len(score))}
    for kind in (2, 3):
        r = rec[rec["kind"] == kind]
        total = covered = 0
        touched = 0
        for t0, t1, sm in zip(r["t0"].astype(np.int64), r["t1"].astype(np.int64), r["sm"]):
            total += t1 - t0
            iv = by_sm.get(int(sm))
            if iv is None:
                continue
            ov = np.clip(np.minimum(iv[:, 1], t1) - np.maximum(iv[:, 0], t0), 0, None).sum()
            covered += int(ov)
            touched += ov > 0
        out[KINDS[kind]] = {"ctas": int(len(r)), "time_share_beside_score": covered / total if total else None,
                            "cta_share_beside_score": touched / len(r) if len(r) else None,
                            "mean_cta_us": total / len(r) / 1e3 if len(r) else None}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--streams", type=int, default=6)
    ap.add_argument("--out", default=None, help="write the report (JSON) here as well")
    args = ap.parse_args()

    import torch
    from hgrnet_b200 import _cabi, ops
    from hgrnet_b200.stream import EvalStream

    lib = _cabi.load()
    if not hasattr(lib, "hgr_placement_attach"):
        raise SystemExit("%s is not a placement build: tools/build_variant.sh placement -DHGR_PLACEMENT "
                         "\"score_pair.cu aggregate_norm.cu topk_merge.cu\"" % _cabi.LIB_PATH)
    attach = lib.hgr_placement_attach
    attach.restype = ctypes.c_int
    attach.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p]

    B, C, D, K = 512, 21841, 1024, 20
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    # three bank copies (134 MB > L2), rotated per slot as in bench.py
    banks = [ops.normalize_rows(torch.randn(C, D, device=dev, generator=g)) for _ in range(3)]
    slots = 2 * args.streams
    es = EvalStream(banks[0], batch=B, K=K, slots=slots, streams=args.streams, banks=banks, host_io=False,
                    feat_dtype=torch.bfloat16)
    for s in range(slots):
        es.dev_feats[s].copy_(torch.randn(B, D, device=dev, generator=g).to(torch.bfloat16))
        es.dev_labels[s].copy_(torch.randint(0, C, (B,), device=dev, generator=g, dtype=torch.int32))
    for i in range(4 * slots):   # warm-up
        es.step(i % slots)
    es.end()
    torch.cuda.synchronize()

    ctas_per_step = 2 * 148 + 64 + 128   # upper bound: scoring CTAs, normalise CTAs, merge CTAs
    cap = ctas_per_step * args.steps
    rec = torch.zeros(cap * REC.itemsize, dtype=torch.uint8, device=dev)
    n = torch.zeros(1, dtype=torch.int32, device=dev)
    chunks = torch.zeros(2, dtype=torch.int64, device=dev)
    _cabi.check(attach(rec.data_ptr(), n.data_ptr(), cap, chunks.data_ptr()))
    es.begin()
    for i in range(args.steps):
        es.step(i % slots)
    es.end()
    torch.cuda.synchronize()
    _cabi.check(attach(None, None, 0, None))

    count = min(int(n.item()), cap)
    recs = np.frombuffer(rec.cpu().numpy().tobytes(), dtype=REC)[:count]
    report = {"workload": "cfg 2 through EvalStream: B = %d, C = %d, D = %d, K = %d, bf16 resident features" % (B, C, D, K),
              "streams": args.streams, "steps": args.steps, "records": count, "dropped": int(n.item()) - count,
              "gpu": torch.cuda.get_device_name(dev), "footprint": ops.score_topk_footprint(B, C, D, K)}
    ts = np.unique(np.concatenate([recs["t0"], recs["t1"]]))
    report["timer_step_ns"] = int(np.diff(ts).min()) if len(ts) > 1 else None   # %globaltimer resolution seen
    report.update(overlap_report(recs))
    ch = chunks.tolist()
    report["topk_chunks"] = {"scanned": ch[0], "not_roomy": ch[1], "share_not_roomy": ch[1] / ch[0] if ch[0] else None}
    line = json.dumps(report)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
