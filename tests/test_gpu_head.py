"""GPU parity of the drop-in ``tree_model`` / ``test()`` surface against the golden fixtures that were
produced by running the UNMODIFIED reference (oracle/gen_golden.py)."""
from __future__ import annotations

import os
import random
import re

import numpy as np
import pytest
import torch

from oracle import cases, hgr_oracle as orc
from tests.util import bf16_input_atol, compare_topk, hits_from_idx, row_rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _opts(tmp_path, **kw):
    from hgrnet_b200.flags import parse_args
    o = parse_args([])
    o.device = 0
    o.folder = str(tmp_path / "out")
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _model(spec, tmp_path, table, test_ids, **optkw):
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import Hierarchy
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens
    h = Hierarchy(cases.tree_edges(spec["levels"], spec["tree_seed"]))
    enc = TableEncoder(table).to(DEV)
    m = tree_model(_opts(tmp_path, **optkw), h.nodes, [h.nodes[i] for i in test_ids], clip_model=enc, hierarchy=h,
                   node_tokens=node_id_tokens(len(h)))
    return m.to(DEV), h


def _ratios(line):
    return [float(x) for x in re.findall(r":(-?\d+\.\d+)", line)]


@pytest.mark.parametrize("spec", cases.EVAL_CASES, ids=[s["name"] for s in cases.EVAL_CASES])
def test_eval_matches_reference_run(spec, tmp_path, golden, golden_dir, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from hgrnet_b200 import evaluate
    from hgrnet_b200.synthetic import FeatureLoader
    n_nodes = sum(spec["levels"])
    test_ids = cases.test_ids(spec, n_nodes)
    table = cases.text_table(spec, n_nodes)
    model, h = _model(spec, tmp_path, table, test_ids, weights="equal")
    g = golden["eval"][spec["name"]]
    z = np.load(os.path.join(golden_dir, spec["name"] + ".npz"))
    batches = cases.eval_batches(spec, test_ids)

    # update_classifier (clip_tree.py:318-325): bank rows vs the reference's zsl_weights
    model.update_classifier()
    step = max(1, n_nodes // 16)
    got = model.zsl_weights[::step].float().cpu()
    ref = torch.from_numpy(z["bank_rows"])
    assert (got - ref).abs().max() <= 2 ** -8 * ref.abs().max()      # bf16 bank: half-ulp of the largest element
    # the test-class bank: the same rows, written by the same pass, in the fixed pseudo-random order `_bank_order`
    assert sorted(model._bank_order.tolist()) == sorted(test_ids)
    assert model._bank_order.tolist() != sorted(test_ids) or len(test_ids) < 3
    assert torch.equal(model.bank_test, model.zsl_weights[model._bank_order])
    assert torch.equal(model._test_index_i32.long(), model._bank_order)

    # forward (clip_tree.py:328-333): dense logits of batch 0 vs the reference's
    logits = model(batches[0][0].to(DEV), None)
    assert logits.shape == (spec["B"], n_nodes) and logits.dtype == torch.float32
    torch.testing.assert_close(logits[:4].cpu(), torch.from_numpy(z["logits0_rows"]), rtol=1e-3,
                               atol=bf16_input_atol(spec["D"]))

    # fused score_topk per batch vs the reference's top-20 ids (main.py:136-141)
    obank = orc.normalize_rows(table)
    hits = torch.zeros(5, dtype=torch.int64, device=DEV)
    ties = 0
    for b, (feats, label) in enumerate(batches):
        tg = torch.full((feats.shape[0],), label, dtype=torch.long, device=DEV)
        val, idx = model.score_topk(feats.to(DEV), tg, hits=hits)
        ref_logits = orc.forward_logits(feats, obank)[:, test_ids]
        assert np.array_equal(orc.eval_hits(orc.forward_logits(feats, obank), torch.tensor(test_ids),
                                            torch.full((feats.shape[0],), label))[0].t().numpy(), z["pred"][b])
        ties += compare_topk(val, idx, ref_logits, test_ids, 20, rtol=1e-3, atol=bf16_input_atol(spec["D"]))
    want = [g["hits"][str(k)] for k in (1, 2, 5, 10, 20)]
    assert all(abs(a - b) <= ties for a, b in zip(hits.tolist(), want)), (hits.tolist(), want, ties)

    # the whole re-hosted test() loop vs the line printed by the reference's main.test (main.py:205-216)
    opts = model.opts
    opts.print_freq = 1000
    loader = FeatureLoader([f for f, _ in batches], [l for _, l in batches])
    line = evaluate.test(opts, model, DEV, loader=loader).strip()
    if ties == 0:
        assert line[: line.index(" hit_ratio")] == g["line"][: g["line"].index(" hit_ratio")]
    mine, ref = _ratios(line), _ratios(g["line"])
    slack = 100.0 * (ties + 2) / g["num_sample"]
    assert len(mine) == len(ref) == 8
    assert all(abs(a - b) <= slack + 0.011 for a, b in zip(mine, ref)), (line, g["line"])
    assert os.path.exists(model.save_path + "arugements.log") and os.path.exists("equal.txt")


@pytest.mark.parametrize("spec", cases.OM_CASES, ids=[s["name"] for s in cases.OM_CASES])
def test_om_step_matches_reference_run(spec, tmp_path, golden, golden_dir):
    n_nodes = sum(spec["levels"])
    table = cases.text_table(spec, n_nodes, normalize=False)
    model, h = _model(spec, tmp_path, table, cases.test_ids(spec, n_nodes), **spec["opts"])
    g = golden["om"][spec["name"]]
    z = np.load(os.path.join(golden_dir, spec["name"] + ".npz"))
    img = cases.image_feats(spec).to(DEV).requires_grad_(True)
    targets = torch.full((spec["B"],), spec["target"], dtype=torch.long, device=DEV)
    random.seed(spec["sample_seed"])
    o = spec["opts"]
    loss = model.train_batch(img, targets, o.get("training_method", "OM"), o.get("sample_strategy", "topk"))
    assert isinstance(loss, float)
    assert len(model.last_losses) == g["T"]
    np.testing.assert_allclose(model.last_losses, g["losses"], rtol=2e-3)
    assert abs(loss - g["loss"]) <= 1e-3 * abs(g["loss"])          # north_star: loss within 1e-3 relative

    def rel(a, b):
        return float((a - b).norm() / b.norm())

    enc = model.clip_model
    d_text = enc.text_table.grad.cpu()
    rows = torch.from_numpy(z["d_text_rows"])
    mask = torch.ones(n_nodes, dtype=torch.bool)
    mask[rows] = False
    assert d_text[mask].abs().max() == 0                               # only sampled classes receive gradient
    assert rel(d_text[rows], torch.from_numpy(z["d_text"])) < 1e-2
    assert rel(img.grad.cpu(), torch.from_numpy(z["d_x"])) < 1e-2
    # per row too: the global measure would pass with one sampled row lost
    assert row_rel_err(d_text[rows], torch.from_numpy(z["d_text"])) < 1e-2
    assert row_rel_err(img.grad.cpu(), torch.from_numpy(z["d_x"])) < 1e-2
    assert abs(float(enc.logit_scale.grad) - float(z["d_log_scale"])) <= 5e-3 * abs(float(z["d_log_scale"])) + 1e-6
    if o["weights"] == "adaptive":
        assert model.layer_weight.grad is not None and model.layer_weight.grad.abs().sum() > 0
        assert "layer_weight" in dict(model.named_parameters())

    # grads accumulate over steps (the reference never calls zero_grad, SURVEY.md section 0)
    g1 = enc.text_table.grad.clone()
    random.seed(spec["sample_seed"])
    model.train_batch(img, targets, o.get("training_method", "OM"), o.get("sample_strategy", "topk"))
    torch.testing.assert_close(enc.text_table.grad, 2 * g1, rtol=1e-5, atol=1e-8)


def test_get_contra_and_get_weights_surface(tmp_path, golden):
    spec = cases.OM_CASES[1]
    n_nodes = sum(spec["levels"])
    model, h = _model(spec, tmp_path, cases.text_table(spec, n_nodes), cases.test_ids(spec, n_nodes), **spec["opts"])
    for key, want in golden["get_weights"].items():
        if key == "layer_weight":
            continue
        method, n = key.rsplit("_", 1)
        got = model.get_weights(method, int(n))
        assert got.device.type == "cuda"
        np.testing.assert_allclose(got.detach().cpu().numpy(), want, rtol=1e-6)
    np.testing.assert_allclose(model.layer_weight.detach().cpu().numpy(), golden["get_weights"]["layer_weight"], rtol=1e-6)
    random.seed(5)
    target = spec["target"]
    parents = h.c2p[target] + [target]
    ids, labels = model.get_contra("topk", target, 16, depth=2, parents=parents)
    assert ids.dtype == torch.long and ids.device.type == "cuda" and labels.shape == (16,)
    assert ids.tolist() == golden["om"][spec["name"]]["compare_idx"][0]
    assert int(labels[0]) == golden["om"][spec["name"]]["labels"][0]


def test_main_cli_runs_eval_and_training_on_synthetic_data(tmp_path, monkeypatch, capsys):
    """`python main.py --train False ...` / `--train True ...` with the reference's flags (README.md:48-49,64)."""
    monkeypatch.chdir(tmp_path)
    import importlib
    import sys
    sys.modules.pop("main", None)
    main = importlib.import_module("main")
    assert os.path.dirname(os.path.abspath(main.__file__)) == os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    common = ["--hgr_synthetic", "6,30,200", "--folder", str(tmp_path / "o"), "--test_batch_size", "96",
              "--batch_size", "32", "--print_freq", "4"]
    main.main(["--train", "False", "--weights", "equal"] + common)
    out = capsys.readouterr().out
    assert "Direct testing." in out and "Top@1(%):" in out and "point_ratio(%):" in out
    main.main(["--train", "True", "--epochs", "1", "--weights", "adaptive", "--out_ratio", "0.5", "--test_after_train"] + common)
    out = capsys.readouterr().out
    assert "loss:" in out and "Model saved." in out and "Top@20(%):" in out


@pytest.mark.parametrize("permute,mode", [(True, "chain"), (False, "chain"), (True, "family")])
def test_update_classifier_chain_bank_matches_oracle(tmp_path, permute, mode):
    """north_star's hierarchy-aggregated bank (`opts.hgr_bank = 'chain'`): row c = normalize(sum_j w_j * E[n_j]) over the
    last ceil(out_ratio * len) nodes of c2p[c] + [c], deepest first, weighted like the OM loop weights its levels
    (clip_tree.py:232-237, :198-219).  Model-level check of kernel (1)'s CSR path against the oracle's restatement,
    and of the fused scorer on that bank."""
    spec = cases.EVAL_CASES[0]
    n_nodes = sum(spec["levels"])
    test_ids = cases.test_ids(spec, n_nodes)
    table = cases.text_table(spec, n_nodes, normalize=False)
    model, h = _model(spec, tmp_path, table, test_ids, weights="increasing", out_ratio=0.5, in_ratio=0.25, hgr_bank=mode,
                      hgr_permute_bank=permute)
    model.update_classifier()
    from hgrnet_b200.levels import level_weights
    rp, col, w = h.chain_csr(0.5, lambda n: level_weights("increasing", n, None).numpy(),
                             include_children=mode == "family", child_weight=0.25)
    assert int(rp[-1]) > n_nodes                                   # rows really aggregate several nodes
    if mode == "family":                                           # the children of node 0 share a weight of in_ratio
        kids = h.p2c[0]
        row0 = list(zip(col[rp[0]:rp[1]].tolist(), w[rp[0]:rp[1]].tolist()))
        assert kids and abs(sum(x for c_, x in row0 if c_ in kids) - 0.25) < 1e-6
    want = orc.aggregate_normalize(table, rp.tolist(), col.tolist(), w.tolist())
    got = model.zsl_weights.float().cpu()
    assert (got - want).abs().max() <= 2 ** -8 * want.abs().max()
    assert torch.equal(model.bank_test, model.zsl_weights[model._bank_order])
    if not permute:
        assert model._bank_order.tolist() == test_ids
    feats, label = cases.eval_batches(spec, test_ids)[0]
    tg = torch.full((feats.shape[0],), label, dtype=torch.long, device=DEV)
    hits = torch.zeros(5, dtype=torch.int64, device=DEV)
    val, idx = model.score_topk(feats.to(DEV), tg, hits=hits)
    ref_logits = orc.forward_logits(feats, want)[:, test_ids]
    compare_topk(val, idx, ref_logits, test_ids, 20, rtol=1e-3, atol=2 * bf16_input_atol(spec["D"]))
    assert hits.tolist() == hits_from_idx(idx, tg.cpu())


@pytest.mark.parametrize("feat_dtype", [torch.float32, torch.float16])
def test_eval_stream_matches_direct_calls(tmp_path, feat_dtype):
    """hgrnet_b200.stream.EvalStream (what bench.py's `value` / `e2e` run): graph-replayed batches on several streams,
    host features in fp32 or fp16, must give the hit counters and top-20 of direct score_topk calls (main.py:131-148)."""
    spec = cases.EVAL_CASES[0]
    n_nodes = sum(spec["levels"])
    test_ids = cases.test_ids(spec, n_nodes)
    table = cases.text_table(spec, n_nodes)
    model, h = _model(spec, tmp_path, table, test_ids, weights="equal")
    model.update_classifier()
    batches = cases.eval_batches(spec, test_ids)
    B = batches[0][0].shape[0]
    es = model.make_eval_stream(batch=B, slots=4, streams=3, feat_dtype=feat_dtype)
    want = torch.zeros(5, dtype=torch.int64, device=DEV)
    es.begin()
    n = 0
    for rep in range(3):
        for i, (feats, label) in enumerate(batches):
            if feats.shape[0] != B:
                continue
            s = n % es.slots
            if n >= es.slots:
                es.synchronize()                       # the slot's previous batch has been consumed
            es.host_feats[s].copy_(feats.to(feat_dtype))
            es.host_labels[s].fill_(label)
            es.step(s)
            tg = torch.full((B,), label, dtype=torch.long, device=DEV)
            v, ix = model.score_topk(feats.to(feat_dtype).to(DEV), tg, hits=want)
            if rep == 0:
                es.synchronize()
                assert torch.equal(es.idx[s], ix)
                torch.testing.assert_close(es.val[s], v, rtol=0, atol=0)
            n += 1
    es.end()
    assert es.hit_counts() == want.tolist() and n >= 3
