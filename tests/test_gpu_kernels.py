"""GPU parity tests of the CUDA kernels, through the C ABI (``hgrnet_b200.ops`` -> libhgr_b200.so),
against the fp32 CPU oracle (``oracle/hgr_oracle.py``) on identical seeded inputs."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import hgr_oracle as orc
from tests.util import compare_topk, hits_from_idx, oracle_hits

pytestmark = pytest.mark.gpu

ops = None
IMPLS = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops, IMPLS
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from hgrnet_b200 import ops as _ops
    ops = _ops
    IMPLS = {"simt": ops.HGR_IMPL_SIMT, "tcgen05": ops.HGR_IMPL_TCGEN05, "tcgen05_exact": ops.HGR_IMPL_TCGEN05_EXACT,
             "tcgen05_sketch": ops.HGR_IMPL_TCGEN05_SKETCH}
    yield
    torch.cuda.synchronize()


def _emb(n, d, seed, normalize=True):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    if normalize:
        x = x / x.norm(dim=-1, keepdim=True)
    return x.to(torch.bfloat16).float()


DEV = "cuda:0"


# --------------------------------------------------------------------------- kernel (1)
@pytest.mark.parametrize("n,d", [(1, 8), (7, 24), (33, 512), (1110, 1024), (300, 520), (64, 2048), (5, 2056), (3, 4096)])
@pytest.mark.parametrize("in_dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_normalize_identity_matches_update_classifier(n, d, in_dtype):
    """identity CSR == `text_feats / text_feats.norm(dim=-1, keepdim=True)` (clip_tree.py:323)."""
    e = (_emb(n, d, 7, normalize=False) * 0.3).to(in_dtype)
    want = orc.normalize_rows(e.float())
    got32, norm = ops.aggregate_normalize(e.to(DEV), out_dtype=torch.float32, return_norm=True)
    assert torch.allclose(got32.cpu(), want, rtol=2e-6, atol=1e-7)
    assert torch.allclose(norm.cpu(), e.float().norm(dim=-1), rtol=2e-6)
    got16 = ops.aggregate_normalize(e.to(DEV), out_dtype=torch.bfloat16)
    # bf16 output: equal to the rounded oracle except where the fp32 value sits on a rounding boundary
    ref16 = want.to(torch.bfloat16)
    diff = (got16.cpu().float() - ref16.float()).abs()
    assert (diff <= ref16.float().abs() * 2 ** -7 + 1e-30).all()
    assert int((got16.cpu() != ref16).sum()) <= max(2, int(1e-3 * ref16.numel()))


@pytest.mark.parametrize("d", [8, 64, 520, 1024, 2048, 2056, 4096])
def test_aggregate_general_csr_and_row_map(d):
    n_src, n_rows = 500, 211
    rng = np.random.RandomState(3)
    e = _emb(n_src, d, 9, normalize=False)
    counts = rng.randint(0, 9, size=n_rows)
    counts[0] = 1
    counts[counts == 0] = 1
    rowptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    col = rng.randint(0, n_src, size=rowptr[-1]).astype(np.int32)
    w = rng.rand(rowptr[-1]).astype(np.float32) + 0.1
    want = orc.aggregate_normalize(e, rowptr, col, w)
    t = lambda a: torch.from_numpy(a).to(DEV)
    got = ops.aggregate_normalize(e.to(DEV), t(rowptr), t(col), t(w), out_dtype=torch.float32)
    assert torch.allclose(got.cpu(), want, rtol=1e-5, atol=1e-6)
    # no weights == all ones
    want1 = orc.aggregate_normalize(e, rowptr, col, np.ones_like(w))
    got1 = ops.aggregate_normalize(e.to(DEV), t(rowptr), t(col), None, out_dtype=torch.float32)
    assert torch.allclose(got1.cpu(), want1, rtol=1e-5, atol=1e-6)
    # row_map: fused gather of the test classes (main.py:136 moved to bank-build time)
    sel = rng.permutation(n_rows)[:77].astype(np.int32)
    got_sel = ops.aggregate_normalize(e.to(DEV), t(rowptr), t(col), t(w), row_map=t(sel), out_dtype=torch.float32)
    assert torch.equal(got_sel, got[torch.from_numpy(sel).long().to(DEV)])
    got_id = ops.aggregate_normalize(e.to(DEV), row_map=t(sel), out_dtype=torch.float32)
    assert torch.allclose(got_id.cpu(), orc.normalize_rows(e)[sel], rtol=2e-6, atol=1e-7)


def test_aggregate_empty_and_errors():
    e = torch.zeros(0, 64, device=DEV)
    assert ops.aggregate_normalize(e).shape == (0, 64)
    from hgrnet_b200._cabi import HgrError
    with pytest.raises(HgrError):
        ops.aggregate_normalize(torch.zeros(4, 12, device=DEV))  # D % 8 != 0
    with pytest.raises(ValueError):
        ops.aggregate_normalize(torch.zeros(4, 16))  # CPU tensor: no CPU path


# --------------------------------------------------------------------------- dense logits
@pytest.mark.parametrize("impl", ["simt", "tcgen05"])
@pytest.mark.parametrize("B,C,D", [(64, 1000, 1024), (37, 313, 256), (1, 16, 64), (129, 4097, 520), (300, 777, 8),
                                   (256, 257, 1024),
                                   # the OM backward's GEMMs: M = U over 12-18 row tiles, N = D, K = B or U
                                   (3000, 1024, 256), (4369, 1024, 264), (256, 1024, 3000), (1024, 2731, 1024)])
def test_logits_dense_matches_forward(impl, B, C, D):
    """`feats @ zsl_weights.T` (clip_tree.py:331) / scaled training logits (:263).  Also per element against float64:
    the products of bf16 inputs are exact in fp32 and D of them are summed in fp32 (<= D 2^-24 of the absolute sum),
    then scaled (2^-24); doubled, |got - ref| <= (D + 2) 2^-23 scale |x| @ |w|."""
    x, w = _emb(B, D, 1), _emb(C, D, 2)
    want = x @ w.T
    ref = x.double() @ w.double().T
    mag = x.double().abs() @ w.double().abs().T
    for scale in (1.0, 14.285714):
        got = ops.logits_dense(x.to(DEV).bfloat16(), w.to(DEV).bfloat16(), scale=scale, impl=IMPLS[impl])
        torch.testing.assert_close(got.cpu(), want * scale, rtol=1e-4, atol=2e-5)
        err = (got.cpu().double() - scale * ref).abs()
        bnd = (D + 2) * 2.0 ** -23 * scale * mag
        assert (err <= bnd).all(), "%d elements outside the bound" % int((err > bnd).sum())


# --------------------------------------------------------------------------- kernel (2)
SHAPES = [
    (64, 1000, 1024),    # BASELINE cfg 1
    (37, 313, 256),      # ragged
    (1, 16, 64),         # single row, single unit
    (5, 5, 64),          # C < K
    (129, 4097, 520),    # two row tiles, D not a multiple of 64, C not a multiple of 16
    (512, 2731, 1024),   # one rank's shard of cfg 5 at 8 GPUs
    (300, 33, 128),
]


@pytest.mark.parametrize("impl", ["simt", "tcgen05", "tcgen05_exact", "tcgen05_sketch"])
@pytest.mark.parametrize("B,C,D", SHAPES)
def test_score_topk_matches_oracle(impl, B, C, D):
    K = 20
    x, w = _emb(B, D, 11), _emb(C, D, 12)
    col_id = torch.from_numpy(np.random.RandomState(5).permutation(10 * C)[:C].astype(np.int32))
    targets = col_id[torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(3))]
    hits = ops.new_hits(DEV)
    xn = ops.normalize_rows(x.to(DEV))
    val, idx = ops.score_topk(xn, w.to(DEV).bfloat16(), col_id=col_id.to(DEV), targets=targets.to(DEV), K=K, hits=hits,
                              impl=IMPLS[impl])
    # oracle on the same bf16 inputs the kernel saw
    logits = xn.float().cpu() @ w.T
    ties = compare_topk(val, idx, logits, col_id, K)
    mine = hits_from_idx(idx, targets)
    assert hits.tolist() == mine, "device hit counters disagree with the returned ids"
    want = oracle_hits(logits, col_id, targets)
    assert all(abs(a - b) <= ties for a, b in zip(mine, want)), (mine, want, ties)
    # hits accumulate across calls
    ops.score_topk(xn, w.to(DEV).bfloat16(), col_id=col_id.to(DEV), targets=targets.to(DEV), K=K, hits=hits, impl=IMPLS[impl])
    assert hits.tolist() == [2 * h for h in mine]


@pytest.mark.parametrize("K", [1, 5, 8, 20, 32])
def test_score_topk_k_values_and_id_base(K):
    B, C, D = 70, 900, 256
    x, w = _emb(B, D, 21), _emb(C, D, 22)
    xn = ops.normalize_rows(x.to(DEV))
    logits = xn.float().cpu() @ w.T
    for impl in ("simt", "tcgen05"):
        val, idx = ops.score_topk(xn, w.to(DEV).bfloat16(), id_base=1000, K=K, scale=14.285714, impl=IMPLS[impl])
        compare_topk(val / 14.285714, idx, logits, torch.arange(C) + 1000, K)


def test_score_topk_tie_order_is_value_desc_then_row_asc():
    """Duplicate bank rows produce exact ties: the lower bank row must come first, on every implementation."""
    B, C, D = 130, 600, 128
    x = _emb(B, D, 31)
    w = _emb(C // 2, D, 32).repeat(2, 1)  # row c and row c + C/2 are identical
    xn = ops.normalize_rows(x.to(DEV))
    outs = []
    for impl in ("simt", "tcgen05_exact", "tcgen05_sketch", "tcgen05"):
        val, idx = ops.score_topk(xn, w.to(DEV).bfloat16(), K=20, impl=IMPLS[impl])
        v, i = val.cpu(), idx.cpu().long()
        same = v[:, :-1] == v[:, 1:]
        assert (i[:, :-1][same] < i[:, 1:][same]).all()
        assert same.any()
        outs.append((v, i))
    # the tcgen05 epilogues see bit-identical accumulators: identical lists, ties included
    assert torch.equal(outs[1][1], outs[2][1]) and torch.equal(outs[1][0], outs[2][0])
    assert torch.equal(outs[1][1], outs[3][1]) and torch.equal(outs[1][0], outs[3][0])


@pytest.mark.parametrize("kind", ["clustered", "ascending", "equal", "dups", "zeros"])
@pytest.mark.parametrize("B,C,D", [(130, 700, 256), (512, 21841, 1024), (4096, 2731, 1024)])
def test_hostile_bank_orders(kind, B, C, D):
    """Banks that break the 'rows in random order' assumption of narrow lists -- siblings adjacent and similar (the
    reference's `nodes` order is graph order), logits rising along the bank, all-equal rows, 40-fold duplicates, zero
    padding.  The production kernel (certificate + exact repair) and the floor-sketch kernel (exact by construction)
    must both return the oracle's top-20 (main.py:136-138), ties resolved by ascending bank row."""
    from tests.util import hostile_bank, hostile_queries
    w = hostile_bank(C, D, kind).to(DEV)
    xn = hostile_queries(w, B, kind)
    logits = (xn.float() @ w.float().T).cpu()
    impls = ["tcgen05_sketch"] if (kind in ("clustered", "ascending", "dups") and B * C > 1e6) else ["tcgen05_sketch", "tcgen05"]
    ref_v, ref_i = ops.score_topk(xn, w, K=20, impl=IMPLS["simt"])
    for impl in impls:      # (the production kernel's repair of a whole hostile cfg-2 bank takes ~1 s: small shape only)
        val, idx = ops.score_topk(xn, w, K=20, impl=IMPLS[impl])
        compare_topk(val, idx, logits, torch.arange(C), 20)
        if kind == "equal":                        # exact ties everywhere: the documented order decides, on every path
            assert torch.equal(idx, ref_i), impl


def test_score_topk_implementations_agree_at_cfg2_size():
    """BASELINE cfg 2 (B=512, C=21,841, D=1024): tcgen05 vs CUDA-core path vs fp32 oracle."""
    B, C, D, K = 512, 21841, 1024, 20
    x, w = _emb(B, D, 41), _emb(C, D, 42)
    xn = ops.normalize_rows(x.to(DEV))
    wb = w.to(DEV).bfloat16()
    targets = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(4)).int()
    h1, h2 = ops.new_hits(DEV), ops.new_hits(DEV)
    v1, i1 = ops.score_topk(xn, wb, targets=targets.to(DEV), K=K, hits=h1, impl=IMPLS["tcgen05"])
    v2, i2 = ops.score_topk(xn, wb, targets=targets.to(DEV), K=K, hits=h2, impl=IMPLS["simt"])
    logits = xn.float().cpu() @ w.T
    t1 = compare_topk(v1, i1, logits, torch.arange(C), K)
    t2 = compare_topk(v2, i2, logits, torch.arange(C), K)
    assert (i1 != i2).any(1).sum() <= t1 + t2
    assert h1.tolist() == hits_from_idx(i1, targets)


@pytest.mark.parametrize("B,C", [(512, 21841), (1024, 10450)])
def test_speculative_lists_are_certified_or_rescanned_exactly(B, C):
    """At cfg 2 size a row is split over 37 lists (18 lists of a row-tile-aligned schedule in the second case), so
    the production kernel keeps SPECULATIVE 8-entry lists.  (a) random bank order: every row certifies, nothing is
    repaired; (b) an adversarial bank whose best classes sit in adjacent rows overflows single lists: the merge must
    detect it and repair those rows exactly (re-scan of the doubtful lists' column ranges)."""
    D, K = 1024, 20
    x, w = _emb(B, D, 51), _emb(C, D, 52)
    xn = ops.normalize_rows(x.to(DEV))
    v0, i0 = ops.score_topk(xn, w.to(DEV).bfloat16(), K=K, impl=IMPLS["tcgen05"])
    assert ops.last_rescan_count(DEV) == 0
    v1, i1 = ops.score_topk(xn, w.to(DEV).bfloat16(), K=K, impl=IMPLS["tcgen05_exact"])
    assert torch.equal(i0, i1) and torch.equal(v0, v1)          # speculation never changes the result
    # adversarial: rows 5000..5039 of the bank are all close to the mean image direction
    w2 = w.clone()
    mean_dir = x.mean(0)
    mean_dir = mean_dir / mean_dir.norm()
    noise = _emb(40, D, 53)
    r0 = C // 4 + 37
    w2[r0:r0 + 40] = ((mean_dir[None, :] * 3 + noise) / (mean_dir[None, :] * 3 + noise).norm(dim=-1, keepdim=True)
                      ).to(torch.bfloat16).float()
    v2, i2 = ops.score_topk(xn, w2.to(DEV).bfloat16(), K=K, impl=IMPLS["tcgen05"])
    rescans = ops.last_rescan_count(DEV)
    assert rescans > 0, "the adversarial bank should overflow at least one speculative list"
    logits = xn.float().cpu() @ w2.T
    compare_topk(v2, i2, logits, torch.arange(C), K)
    v3, i3 = ops.score_topk(xn, w2.to(DEV).bfloat16(), K=K, impl=IMPLS["tcgen05_exact"])
    assert (i2 != i3).any(1).sum() <= max(2, B // 256)          # repaired rows use CUDA-core sums: near-ties may swap


def test_score_topk_empty_and_bad_args():
    from hgrnet_b200._cabi import HgrError
    x = torch.zeros(4, 64, device=DEV, dtype=torch.bfloat16)
    val, idx = ops.score_topk(x, torch.zeros(0, 64, device=DEV, dtype=torch.bfloat16), K=20)
    assert torch.isinf(val).all() and (idx == -1).all()
    v, i = ops.score_topk(torch.zeros(0, 64, device=DEV, dtype=torch.bfloat16), x, K=20)
    assert v.shape == (0, 20)
    with pytest.raises(HgrError):
        ops.score_topk(x, x, K=33)
    with pytest.raises(HgrError):
        ops.score_topk(x, x, K=20, scale=-1.0)
    with pytest.raises(TypeError):
        ops.score_topk(x.float(), x, K=20)
    with pytest.raises(HgrError, match="320"):         # more lists per row than the merge kernels hold
        ops.topk_merge(torch.zeros(321, 4, 7, device=DEV), torch.zeros(321, 4, 7, dtype=torch.int32, device=DEV))


# --------------------------------------------------------------------------- merge
@pytest.mark.parametrize("P,B,K", [(1, 5, 20), (2, 64, 20), (4, 70, 20), (3, 40, 32), (5, 1000, 20), (8, 130, 20), (37, 33, 20),
                                   (128, 9, 7), (129, 9, 20), (320, 5, 7)])
def test_topk_merge_matches_sort(P, B, K):
    g = torch.Generator().manual_seed(P * 100 + B)
    vals = torch.randn(P, B, K, generator=g)
    vals, _ = vals.sort(dim=2, descending=True)
    ids = torch.stack([torch.randperm(P * K, generator=g).reshape(P, K) for _ in range(B)], 1).int()  # unique per row
    # a few empty tails
    vals[0, :, K // 2:] = float("-inf")
    ids[0, :, K // 2:] = -1
    targets = ids[P - 1, :, 0].clone()
    hits = ops.new_hits(DEV)
    v, i = ops.topk_merge(vals.to(DEV), ids.to(DEV), targets=targets.to(DEV), hits=hits)
    flat_v = vals.permute(1, 0, 2).reshape(B, P * K)
    flat_i = ids.permute(1, 0, 2).reshape(B, P * K)
    ov, op = flat_v.topk(K, 1, True, True)
    assert torch.equal(v.cpu(), ov)
    assert torch.equal(i.cpu(), flat_i.gather(1, op))
    assert hits.tolist() == hits_from_idx(i, targets)


# --------------------------------------------------------------------------- kernel (3)
def _ce_oracle(logits, sets, label_pos, weight):
    """clip_tree.py:275-276 per iteration, fp32 torch autograd."""
    lg = logits.clone().requires_grad_(True)
    losses = []
    for ids, lp, w in zip(sets, label_pos, weight):
        sub = lg[:, torch.tensor(ids)]
        l = torch.nn.CrossEntropyLoss()(sub, torch.full((lg.shape[0],), lp)) * w
        l.backward()
        losses.append(l.item())
    return torch.tensor(losses), lg.grad


@pytest.mark.parametrize("B,U,T", [(16, 24, 2), (256, 1500, 17), (24, 700, 12), (3, 9000, 5), (1, 1, 1)])
def test_masked_ce_matches_crossentropy(B, U, T):
    rng = np.random.RandomState(B + U)
    logits = torch.randn(B, U, generator=torch.Generator().manual_seed(U)) * 3
    sets, lps = [], []
    for t in range(T):
        n = int(rng.randint(1, min(U, 257) + 1))
        ids = rng.permutation(U)[:n].tolist()
        sets.append(ids)
        lps.append(int(rng.randint(n)))
    weight = (rng.rand(T).astype(np.float32) + 0.05)
    want_l, want_g = _ce_oracle(logits, sets, lps, weight.tolist())
    set_ptr = np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.int32)
    set_col = np.concatenate(sets).astype(np.int32)
    t = lambda a: torch.from_numpy(np.asarray(a)).to(DEV)
    loss, dl = ops.masked_ce(logits.to(DEV), t(set_ptr), t(set_col), t(np.asarray(lps, np.int32)), t(weight))
    torch.testing.assert_close(loss.cpu(), want_l, rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(dl.cpu(), want_g, rtol=1e-4, atol=1e-7)
    loss2, none = ops.masked_ce(logits.to(DEV), t(set_ptr), t(set_col), t(np.asarray(lps, np.int32)), t(weight),
                                need_grad=False)
    assert none is None and torch.equal(loss2, loss)
