"""Measurements of the rows of SURVEY.md section 8d that are not the bench.py headline:

* cfg 3 -- one OM training step of the head (B=256, D=1024, 12-level 21,841-node hierarchy, out 0.25 / in 0.5,
  adaptive weights, --k 1, num_compare 256, deepest-level target): `tree_model.train_batch` (kernel 1 + dense
  logits + fused masked CE, all T iterations in one launch) vs the reference's per-iteration torch loop on the
  same GPU and on the host CPU;
* kernel (3) alone: microseconds and achieved GB/s against the HBM roofline (algorithmic bytes 8*B*U);
* kernel (1) at bank size (21,841 x 1024): achieved GB/s, identity CSR and a chain-aggregated CSR.
Prints one JSON object; run on the GPU box.
"""
import json
import os
import random
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from hgrnet_b200 import ops
from hgrnet_b200.flags import parse_args
from hgrnet_b200.head import tree_model
from hgrnet_b200.hierarchy import WORDNET_LIKE_21841, synthetic_hierarchy
from hgrnet_b200.levels import level_weights
from hgrnet_b200.synthetic import TableEncoder, node_id_tokens, synthetic_embeddings

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sweep import timeit as graph_us   # per-call microseconds with the interpreter off the path (CUDA graph replay)

DEV = "cuda:0"
HBM = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"] \
    if os.path.exists(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")) else 6650.0


def events(fn, n, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3  # us


def torch_loop_step(model, img, target, device):
    """The reference's OM loop (clip_tree.py:222-281) with stock torch ops on `device` (fp32)."""
    from oracle import hgr_oracle as orc
    enc = model.clip_model
    img_feats = enc.encode_image(img)
    img_n = img_feats / img_feats.norm(dim=-1, keepdim=True)
    img_ = img_n.detach().clone().requires_grad_(True)
    lw = model.layer_weight.detach() if hasattr(model, "layer_weight") else None
    ce = torch.nn.CrossEntropyLoss()
    losses = []
    for (k_loop, m_loop, p_out, depth, parents_in, n_out, n_in) in orc.om_schedule(model.c2p, target, model.opts.out_ratio, model.opts.in_ratio):
        ids, labels = orc.get_contra_topk(model.d2n, p_out, img.shape[0], depth, parents_in, model.opts.k, model.opts.num_compare)
        tf = enc.encode_text(model.node_tokens[torch.tensor(ids, device=device)])
        tf = tf / tf.norm(dim=-1, keepdim=True)
        logits = (img_ @ tf.t()) * enc.logit_scale.exp()
        w_in = orc.get_weights(model.opts.weights, n_in, lw.cpu() if lw is not None else None)
        w_out = orc.get_weights(model.opts.weights, n_out, lw.cpu() if lw is not None else None)
        loss_j = ce(logits, torch.tensor(labels, device=device)) * float(w_in[m_loop]) * float(w_out[k_loop])
        loss_j.backward()
        losses.append(loss_j.item())
    img_feats.backward(img_.grad)
    return sum(losses), len(losses)


def main():
    out = {}
    hier = synthetic_hierarchy(WORDNET_LIKE_21841, seed=1)
    N, D, B = len(hier), 1024, 256
    table = synthetic_embeddings(N, D, 1, normalize=False)
    opts = parse_args([])
    opts.device, opts.folder = 0, "/tmp/hgr_om_bench"
    model = tree_model(opts, hier.nodes, hier.nodes, clip_model=TableEncoder(table).to(DEV), hierarchy=hier,
                       node_tokens=node_id_tokens(N))
    target = N - 1                                     # deepest level: chain of 12 -> T = 17
    img = synthetic_embeddings(B, D, 5, normalize=False).to(DEV).requires_grad_(True)
    targets = torch.full((B,), target, dtype=torch.long, device=DEV)

    def ours():
        random.seed(0)
        return model.train_batch(img, targets, "OM", "topk")

    loss = ours()
    T = len(model.last_losses)
    random.seed(0)
    ref_loss, T_ref = torch_loop_step(model, img, target, DEV)
    us_ours = events(ours, 30)
    us_loop = events(lambda: (random.seed(0), torch_loop_step(model, img, target, DEV)), 10)
    # host CPU (reference torch ops, fp32)
    model_cpu_enc = TableEncoder(table)
    class _M:  # duck-typed view of the model on the CPU
        pass
    m = _M()
    m.clip_model, m.c2p, m.d2n, m.opts, m.node_tokens = model_cpu_enc, model.c2p, model.d2n, model.opts, model.node_tokens.cpu()
    m.layer_weight = model.layer_weight.detach().cpu()
    img_cpu = img.detach().cpu().requires_grad_(True)
    random.seed(0)
    torch_loop_step(m, img_cpu, target, "cpu")
    t0 = time.perf_counter()
    for _ in range(3):
        random.seed(0)
        torch_loop_step(m, img_cpu, target, "cpu")
    us_cpu = (time.perf_counter() - t0) / 3 * 1e6
    out["om_step_cfg3"] = {"B": B, "D": D, "T": T, "loss_ours": loss, "loss_torch_loop": ref_loss,
                           "us_per_step_ours": us_ours, "us_per_step_torch_loop_gpu": us_loop,
                           "us_per_step_torch_loop_cpu": us_cpu, "cpu_threads": torch.get_num_threads(),
                           "speedup_vs_gpu_loop": us_loop / us_ours, "speedup_vs_cpu": us_cpu / us_ours,
                           "note": "encoders are table look-ups here, so this is the head alone (the reference's step is dominated by encode_text)"}

    # ---- kernel (3) alone at cfg-3 shape: union of T=17 sets of <=257 classes
    rng = np.random.RandomState(0)
    U = 3000
    logits = torch.randn(B, U, device=DEV) * 3
    sets = [rng.permutation(U)[:257] for _ in range(17)]
    set_ptr = torch.tensor(np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.int32), device=DEV)
    set_col = torch.tensor(np.concatenate(sets).astype(np.int32), device=DEV)
    lp = torch.tensor(rng.randint(0, 257, 17).astype(np.int32), device=DEV)
    w = torch.rand(17, device=DEV)
    us_ce = graph_us(lambda i: ops.masked_ce(logits, set_ptr, set_col, lp, w))
    bytes_ce = 8.0 * B * U
    out["masked_ce_kernel"] = {"B": B, "U": U, "T": 17, "us": us_ce, "algorithmic_bytes": bytes_ce,
                               "achieved_GBs": bytes_ce / (us_ce * 1e-6) / 1e9, "hbm_peak_GBs": HBM,
                               "frac": bytes_ce / (us_ce * 1e-6) / 1e9 / HBM,
                               "note": "2 launches (CE + loss reduce); latency-bound at this size"}

    # ---- the head's own device work of one cfg-3 step, interpreter and encoder stand-in off the path: normalise the
    # image batch and the union's text rows, tcgen05 logits, fused masked CE, tcgen05 backward (one CUDA graph replay)
    xr = torch.randn(B, D, device=DEV)
    tr = torch.randn(U, D, device=DEV)

    def head_device(i):
        xn_, xnorm_ = ops.normalize_rows(xr, return_norm=True)
        tn_, tnorm_ = ops.normalize_rows(tr, return_norm=True)
        lg_ = ops.logits_dense(xn_, tn_, scale=14.2857)
        _, dl_ = ops.masked_ce(lg_, set_ptr, set_col, lp, w)
        ops.om_backward(dl_, lg_, xn_, xnorm_, tn_, tnorm_, 14.2857)
    us_head = graph_us(head_device)
    out["om_step_cfg3"]["us_head_kernels_per_step"] = us_head
    out["om_step_cfg3"]["note_breakdown"] = ("of the wall clock per step ~0.2 ms is the host-side plan of the step (one call of the library host helper), "
                                             "the head's own kernels take us_head_kernels_per_step; the rest is the "
                                             "stand-in encoder's autograd (a dense 21,841 x 1024 table gradient per step) "
                                             "and three host synchronisations (label, logit scale, losses)")

    # ---- kernel (1) at bank size
    E = synthetic_embeddings(N, D, 2, normalize=False).to(DEV)
    us_id = graph_us(lambda i: ops.aggregate_normalize(E))
    b_id = N * D * 4 + N * D * 2
    Eb = E.bfloat16()
    us_id16 = graph_us(lambda i: ops.aggregate_normalize(Eb))
    b_id16 = N * D * 2 * 2
    rp, col, wt = hier.chain_csr(0.25, lambda n: level_weights("increasing", n).numpy())
    t = lambda a: torch.from_numpy(a).to(DEV)
    rp_d, col_d, w_d = t(rp), t(col), t(wt)
    us_ch = graph_us(lambda i: ops.aggregate_normalize(Eb, rp_d, col_d, w_d))
    nnz = int(rp[-1])
    b_ch = 2 * N * D * 2 + 4 * (nnz + N + 1) + 4 * nnz       # compulsory: every source row once + output + CSR
    out["aggregate_normalize_bank"] = {
        "N": N, "D": D, "hbm_peak_GBs": HBM,
        "identity_fp32_in": {"us": us_id, "bytes": b_id, "GBs": b_id / us_id / 1e3, "frac": b_id / us_id / 1e3 / HBM},
        "identity_bf16_in": {"us": us_id16, "bytes": b_id16, "GBs": b_id16 / us_id16 / 1e3, "frac": b_id16 / us_id16 / 1e3 / HBM},
        "chain_csr_bf16_in": {"us": us_ch, "nnz": nnz, "compulsory_bytes": b_ch, "GBs": b_ch / us_ch / 1e3,
                              "frac": b_ch / us_ch / 1e3 / HBM, "gathered_GBs": (nnz * D * 2 + N * D * 2) / us_ch / 1e3}}
    # ---- row f1: TOR / POR at cfg-2 shape (B=512 rows against 21,841 nodes, chain of 12)
    from hgrnet_b200.evaluate import HierMetrics
    Bt = 512
    xt = ops.normalize_rows(synthetic_embeddings(Bt, D, 7, normalize=False).to(DEV))
    model.update_classifier()
    dense = ops.logits_dense(xt, model.bank_train)           # train columns only (here: every node is a train class)
    hm = HierMetrics(model)
    tt = torch.full((Bt,), target, dtype=torch.int32, device=DEV)
    us_dense = graph_us(lambda i: ops.logits_dense(xt, model.bank_train, out=dense))
    us_fused = events(lambda: hm.update_rows(xt, tt), 50)
    parents = list(model.c2p[target]) + [target]
    depth_t = torch.from_numpy(hier.depth).to(DEV)

    def reference_passes():                                   # main.py:153-176 with stock torch ops on the GPU
        lt = dense[:, model.train_index]
        _ = model.train_index[lt.topk(1, 1, True, True)[1]]
        for p in parents:
            rest = (depth_t != len(model.c2p[p])).nonzero().squeeze(1)
            lk = dense.detach().clone().index_fill(1, rest, -1)[:, model.train_index]
            _ = model.train_index[lk.topk(1, 1, True, True)[1]].squeeze()
    us_ref = events(reference_passes, 5)
    # the metrics WITHOUT the dense matrix: per-level arg-max in the GEMM epilogue over the level-sorted bank
    args, cnt_ = hm.rows_args(), ops.new_hier_counts(DEV)
    us_nodense = graph_us(lambda i: ops.hier_metrics_fused_rows(xt, targets=tt, counts=cnt_, **args))
    out["hier_metrics_f1"] = {"B": Bt, "N": N, "L": len(parents), "us_kernel_plus_host_glue": us_fused,
                              "us_fused_in_gemm_epilogue": us_nodense, "us_dense_logits": us_dense,
                              "us_reference_torch_passes_gpu": us_ref,
                              "speedup_vs_torch_passes": us_ref / us_fused,
                              "note": "reference = L+1 clone/index_fill/gather/topk passes over [B,N] (without its Python "
                                      "BxL loop and without the dense logits they read); ours = HierMetrics.update_rows "
                                      "(GEMM + finish + totals)"}
    # ---- the same row with a REAL-SHAPED train split: 1,000 train classes + their ancestors (ImageNet-1K inside the
    # 21K hierarchy: ~1,900 of 21,841 nodes), test bank = all 21,841 nodes.  What `evaluate.test` runs per batch with
    # the metrics on: fused top-20 head + the per-level arg-max GEMM over the TRAIN rows, against the head alone.
    rs = np.random.RandomState(3)
    deep = [n for n in range(N) if hier.depth[n] >= 5]
    picked = set()
    for n in rs.permutation(deep)[:1000].tolist():
        picked.add(n)
        picked.update(model.c2p[n])
    train_nodes = [hier.nodes[n] for n in sorted(picked)]
    m2 = tree_model(opts, train_nodes, hier.nodes, clip_model=TableEncoder(table).to(DEV), hierarchy=hier,
                    node_tokens=node_id_tokens(N))
    m2.update_classifier()
    hm2 = HierMetrics(m2)
    tgt2 = sorted(picked)[-1]
    lab2 = torch.full((Bt,), tgt2, dtype=torch.int32, device=DEV)
    hits2 = ops.new_hits(DEV)
    args2, cnt2 = hm2.rows_args(), ops.new_hier_counts(DEV)
    us_head = graph_us(lambda i: ops.score_topk(xt, m2.bank_test, col_id=m2._test_index_i32, targets=lab2, K=20, hits=hits2))

    def with_metrics(i):
        ops.score_topk(xt, m2.bank_test, col_id=m2._test_index_i32, targets=lab2, K=20, hits=hits2)
        ops.hier_metrics_fused_rows(xt, targets=lab2, counts=cnt2, **args2)
    us_with = graph_us(with_metrics)
    out["hier_metrics_f1_real_split"] = {
        "B": Bt, "test_classes": int(m2.bank_test.shape[0]), "train_columns": int(m2.bank_train.shape[0]),
        "us_head_alone": us_head, "us_head_plus_metrics": us_with, "ratio": us_with / us_head,
        "note": "kernels of one eval batch (one CUDA graph replay each, same bank every replay: L2-warm); metrics = "
                "hgr_hier_metrics_fused_rows (per-level arg-max in the GEMM epilogue over the train rows)"}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
