"""GPU parity at the FULL sizes of every measured BASELINE configuration, through the C ABI, against the fp32
oracle on identical bf16-valued inputs (tie-aware ids, hit counters, values / loss within 1e-3):

* cfg 5 and its per-rank shards: B = 4096 x C in {21,841, 10,921, 5,461, 2,731}, D = 1024 (main.py:136-147);
* cfg 4: (1024, 10,450, 512);
* cfg 3: the OM step at B = 256, D = 1024, 12-level 21,841-node hierarchy, T = 17 (clip_tree.py:222-281);
* the class-sharded peer exchange with 8 logical ranks at B = 4096, against the ORACLE (not our own 1-GPU result).
"""
from __future__ import annotations

import random

import numpy as np
import pytest
import torch

from oracle import hgr_oracle as orc
from tests.util import compare_topk, hits_from_idx, oracle_hits, row_rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
K = 20


def _emb(n, d, seed, normalize=True):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    if normalize:
        x = x / x.norm(dim=-1, keepdim=True)
    return x.to(torch.bfloat16).float()


def _oracle_logits(xn_dev, w):
    """fp32 `feats @ zsl_weights.T` (clip_tree.py:331) on the host, on the bf16 inputs the kernel saw."""
    return xn_dev.float().cpu() @ w.T


def _check_against_oracle(B, C, D, impl_names=("tcgen05",), seed=0):
    from hgrnet_b200 import ops
    impls = {"tcgen05": ops.HGR_IMPL_TCGEN05, "tcgen05_exact": ops.HGR_IMPL_TCGEN05_EXACT, "simt": ops.HGR_IMPL_SIMT}
    x, w = _emb(B, D, 61 + seed), _emb(C, D, 62 + seed)
    xn = ops.normalize_rows(x.to(DEV))
    wb = w.to(DEV).bfloat16()
    col_id = torch.from_numpy(np.random.RandomState(7).permutation(3 * C)[:C].astype(np.int32))
    targets = col_id[torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(5))]
    logits = _oracle_logits(xn, w)
    want = oracle_hits(logits, col_id, targets)
    outs = []
    for name in impl_names:
        hits = ops.new_hits(DEV)
        val, idx = ops.score_topk(xn, wb, col_id=col_id.to(DEV), targets=targets.to(DEV), K=K, hits=hits, impl=impls[name])
        ties = compare_topk(val, idx, logits, col_id, K)
        mine = hits_from_idx(idx, targets)
        assert hits.tolist() == mine, "device hit counters disagree with the returned ids"
        assert all(abs(a - b) <= ties for a, b in zip(mine, want)), (name, mine, want, ties)
        outs.append((val.cpu(), idx.cpu()))
    for o in outs[1:]:      # the tcgen05 variants see bit-identical accumulators
        assert torch.equal(o[1], outs[0][1]) and torch.equal(o[0], outs[0][0])


@pytest.mark.parametrize("C", [21841, 10921, 5461, 2731])
def test_cfg5_and_its_shards_match_oracle(C):
    """B = 4096: the shape every multi-GPU number runs (full bank at N = 1; a rank's shard at N = 2 / 4 / 8)."""
    _check_against_oracle(4096, C, 1024, ("tcgen05", "tcgen05_exact"))


def test_cfg4_matches_oracle():
    """ImageNet-21K-P split: ~10,450 classes, ViT-B/32 dim 512, batch 1024."""
    _check_against_oracle(1024, 10450, 512, ("tcgen05", "tcgen05_exact"))


@pytest.mark.parametrize("B,C,D", [(512, 21841, 1024), (512, 18278, 1024), (1024, 10021, 512), (256, 21841, 768),
                                   (300, 5000, 640), (4096, 2731, 512)])
def test_other_real_sizes_match_oracle(B, C, D):
    """cfg 2, the reference's real class counts (18,278 / 10,021, SURVEY section 0) and the other CLIP widths."""
    _check_against_oracle(B, C, D)


@pytest.mark.parametrize("certify", ["global", "local"])
def test_class_sharded_exchange_matches_oracle_at_cfg5(certify):
    """8 logical ranks on one GPU, B = 4096, C = 21,841: every rank scores its class shard, scatters its local
    top-20 to the row owners over (here: local) peer memory, owners merge -- compared with the fp32 ORACLE.
    `global`: the production arrangement of ShardedEvalStream (narrow lists certified by the row owner against the
    global K-th value); `local`: exact 20-entry lists per shard."""
    from hgrnet_b200 import ops
    from hgrnet_b200.dist import PeerExchange, exchange_layout, shard_bounds
    dev = torch.device(DEV)
    B, C, D, G = 4096, 21841, 1024, 8
    x, w = _emb(B, D, 71), _emb(C, D, 72)
    xn = ops.normalize_rows(x.to(dev))
    wb = w.to(dev).bfloat16()
    targets = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(9)).int()
    logits = _oracle_logits(xn, w)
    lay = exchange_layout(B, K, G, 4)
    bufs = [ops.peer_alloc(lay["total"])[0] for _ in range(G)]
    try:
        ranks = [PeerExchange(B, K, dev, slots=4, _bases=bufs, _rank=r, _world=G) for r in range(G)]
        bounds = shard_bounds(C, G)
        hits = ops.new_hits(dev)
        shards = [wb[lo:hi].contiguous() for lo, hi in bounds]
        cert = None
        if certify == "global":
            table = ops.shard_table([(s.data_ptr(), 0, s.shape[0], lo) for s, (lo, _) in zip(shards, bounds)], dev)
            repairs = torch.zeros(1, dtype=torch.int32, device=dev)
            cert = (xn, table, repairs)
            assert ops.global_list_len(B, shards[0].shape[0], D, K, C) < K
        for r, px in enumerate(ranks):
            px.scatter(xn, shards[r], bounds[r][0], 0, C_total=C if cert else 0)
        outs = [px.merge(0, targets.to(dev), hits, certify=cert) for px in ranks]
        torch.cuda.synchronize()
        if cert:
            assert int(repairs.item()) == 0
        val = torch.cat([o[0] for o in outs if o is not None])
        idx = torch.cat([o[1] for o in outs if o is not None])
        ties = compare_topk(val, idx, logits, torch.arange(C), K)
        mine = hits_from_idx(idx, targets)
        assert hits.tolist() == mine
        want = oracle_hits(logits, torch.arange(C), targets)
        assert all(abs(a - b) <= ties for a, b in zip(mine, want)), (mine, want, ties)
    finally:
        torch.cuda.synchronize()
        for b in bufs:
            ops.peer_free(b)


def test_cfg3_om_step_matches_oracle(tmp_path):
    """BASELINE cfg 3: OM step, --sample_strategy topk, out 0.25 / in 0.5, adaptive weights, batch 256, dim 1024,
    12-level 21,841-node hierarchy, target on the deepest level (chain of 12 => T = 17).  Loss within 1e-3 relative,
    gradients vs the oracle's autograd restatement of clip_tree.py:222-281."""
    from hgrnet_b200.flags import parse_args
    from hgrnet_b200.head import tree_model
    from hgrnet_b200.hierarchy import scaled_levels, synthetic_hierarchy
    from hgrnet_b200.levels import layer_weight_init
    from hgrnet_b200.synthetic import TableEncoder, node_id_tokens
    N, D, B = 21841, 1024, 256
    h = synthetic_hierarchy(scaled_levels(N), seed=1)
    table = (_emb(N, D, 81, normalize=False) * 0.05).to(torch.bfloat16).float()
    img = _emb(B, D, 82, normalize=False)
    target = max(range(N), key=lambda i: len(h.c2p[i]))
    assert len(h.c2p[target]) + 1 == 12
    o = parse_args([])
    o.device, o.folder = 0, str(tmp_path / "out")
    o.weights, o.out_ratio, o.in_ratio, o.k, o.num_compare, o.weighting, o.scale = "adaptive", 0.25, 0.5, 1, 256, "both", 1.0
    enc = TableEncoder(table).to(DEV)
    model = tree_model(o, h.nodes, h.nodes, clip_model=enc, hierarchy=h, node_tokens=node_id_tokens(N)).to(DEV)
    x = img.to(DEV).requires_grad_(True)
    random.seed(17)
    loss = model.train_batch(x, torch.full((B,), target, dtype=torch.long, device=DEV), "OM", "topk")
    random.seed(17)
    ref = orc.om_step(img, table, torch.tensor(float(np.log(1 / 0.07))), h.c2p, h.d2n, target, out_ratio=0.25,
                      in_ratio=0.5, weights="adaptive", weighting="both", k=1, num_compare=256,
                      layer_weight=layer_weight_init(h.d2n, 1.0))
    assert len(model.last_losses) == len(ref["losses"]) == 17
    np.testing.assert_allclose(model.last_losses, ref["losses"], rtol=2e-3)
    assert abs(loss - ref["loss"]) <= 1e-3 * abs(ref["loss"]), (loss, ref["loss"])

    def rel(a, b):
        return float((a - b).norm() / b.norm())

    d_text = enc.text_table.grad.cpu()
    touched = ref["d_text_raw"].abs().sum(1) > 0
    assert d_text[~touched].abs().max() == 0
    assert rel(d_text[touched], ref["d_text_raw"][touched]) < 1e-2
    assert row_rel_err(d_text[touched], ref["d_text_raw"][touched]) < 1e-2     # every touched row, not just the sum
    # the oracle reports the gradient w.r.t. the NORMALISED image features (clip_tree.py:226,280); chain it through
    # the row normalisation the way `img_feats.backward(img_feats_.grad)` does
    imgf = img.clone().requires_grad_(True)
    (imgf / imgf.norm(dim=-1, keepdim=True)).backward(ref["d_img_n"])
    assert rel(x.grad.cpu(), imgf.grad) < 1e-2
    assert row_rel_err(x.grad.cpu(), imgf.grad) < 1e-2
    assert abs(float(enc.logit_scale.grad) - float(ref["d_log_scale"])) <= 5e-3 * abs(float(ref["d_log_scale"])) + 1e-6
