"""Shared helpers of the test-suite: tie-aware top-k comparison against the fp32 oracle."""
from __future__ import annotations

import numpy as np
import torch

LOGIT_RTOL = 1e-3   # north_star: logits / loss within 1e-3 relative under bf16-in / fp32-accumulate
LOGIT_ATOL = 1e-5


def bf16_input_atol(D):
    """Absolute logit tolerance when the comparison partner saw UNROUNDED fp32 normalised features (the reference
    run behind the golden files) while the kernels see them rounded to bf16 (relative error <= 2^-9 per element of
    both unit vectors): the dot product moves by ~2^-9 * sqrt(2/3) / sqrt(D) (1 sigma); 6x that is the bound used."""
    return 6.0 * 2.0 ** -9 / float(D) ** 0.5


def compare_topk(val, idx, oracle_logits, col_ids, K, rtol=LOGIT_RTOL, atol=LOGIT_ATOL):
    """Compare a device top-K (``val`` [B,K] fp32, ``idx`` [B,K] node ids) with the oracle logits
    ``oracle_logits`` [B,C] (column c belongs to node ``col_ids[c]``).

    Bar (BASELINE.md section 4): ids bit-exact except at ties inside the logit tolerance -- a
    differing id is accepted only if its oracle logit is within tolerance of the oracle's K-th
    value; values within tolerance; list sorted descending.  Returns the number of rows that
    needed the tie rule.
    """
    val = val.detach().cpu().float()
    idx = idx.detach().cpu().long()
    B, C = oracle_logits.shape
    Kv = min(K, C)
    col_ids = torch.as_tensor(col_ids).long()
    pos_of = {int(n): c for c, n in enumerate(col_ids.tolist())}
    ov, oi = oracle_logits.topk(Kv, 1, True, True)
    oid = col_ids[oi]
    # padding when C < K
    if Kv < K:
        assert torch.isinf(val[:, Kv:]).all() and (val[:, Kv:] < 0).all()
        assert (idx[:, Kv:] == -1).all()
    v, i = val[:, :Kv], idx[:, :Kv]
    assert (v[:, :-1] >= v[:, 1:]).all(), "top-k values not sorted descending"
    assert torch.allclose(v, ov, rtol=rtol, atol=atol), "top-k values off: max abs err %g" % (v - ov).abs().max()
    tie_rows = 0
    mism = (i != oid).any(1).nonzero().squeeze(1).tolist()
    for b in mism:
        mine, ref = set(i[b].tolist()), set(oid[b].tolist())
        kth = float(ov[b, -1])
        tol = atol + rtol * abs(kth)
        for n in mine ^ ref:
            assert n in pos_of, "row %d: id %d is not a test class" % (b, n)
            lv = float(oracle_logits[b, pos_of[n]])
            assert abs(lv - kth) <= tol, "row %d: id %d (logit %g) differs outside the tie tolerance of k-th %g" % (b, n, lv, kth)
        # same set but different order: every swapped pair must be a near-tie
        for k in range(Kv):
            if i[b, k] != oid[b, k]:
                lv = float(oracle_logits[b, pos_of[int(i[b, k])]])
                assert abs(lv - float(ov[b, k])) <= atol + rtol * abs(float(ov[b, k])), \
                    "row %d rank %d: order differs outside the tie tolerance" % (b, k)
        tie_rows += 1
    # reported value belongs to the reported id
    gathered = oracle_logits.gather(1, torch.tensor([[pos_of[int(n)] for n in row] for row in i.tolist()]))
    assert torch.allclose(v, gathered, rtol=rtol, atol=atol), "value / id pairs inconsistent"
    return tie_rows


def row_rel_err(got, ref):
    """Largest per-row relative error ``|got_r - ref_r| / |ref_r|`` over the rows of ``ref`` that are not zero; a zero
    row of ``ref`` must be zero in ``got`` too (inf otherwise).  A global Frobenius measure hides a lost row."""
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    rn = ref.norm(dim=1)
    zero = rn == 0
    if (got[zero] != 0).any():
        return float("inf")
    if not (~zero).any():
        return 0.0
    return float(((got - ref).norm(dim=1)[~zero] / rn[~zero]).max())


def hits_from_idx(idx, targets, cuts=(1, 2, 5, 10, 20)):
    idx = idx.detach().cpu().long()
    targets = torch.as_tensor(targets).long().reshape(-1, 1)
    eq = idx == targets
    return [int(eq[:, :k].any(1).sum()) for k in cuts]


def oracle_hits(oracle_logits, col_ids, targets, cuts=(1, 2, 5, 10, 20)):
    K = min(max(cuts), oracle_logits.shape[1])
    oi = oracle_logits.topk(K, 1, True, True)[1]
    return hits_from_idx(torch.as_tensor(col_ids).long()[oi], targets, cuts)


def _unit_bf16(w):
    return (w / w.norm(dim=-1, keepdim=True).clamp_min(1e-12)).to(torch.bfloat16)


def hostile_bank(C, D, kind, seed=3):
    """Class banks whose row order is NOT random (what narrow speculative lists assume):
    clustered -- siblings adjacent and similar (child = parent + noise, rows in tree order, like the reference's `nodes`);
    ascending -- every image's logits rise along the bank;  equal -- all rows identical (every logit of a row ties);
    dups -- 40 copies of every distinct row;  zeros -- mostly zero rows (padding) and a few real ones;  iid -- control."""
    g = torch.Generator().manual_seed(seed)
    if kind == "iid":
        return _unit_bf16(torch.randn(C, D, generator=g))
    if kind == "clustered":
        centers = torch.randn((C + 63) // 64, D, generator=g)
        return _unit_bf16(centers.repeat_interleave(64, 0)[:C] + 0.15 * torch.randn(C, D, generator=g))
    if kind == "ascending":
        base = torch.randn(1, D, generator=g)
        t = torch.linspace(0.0, 1.0, C).unsqueeze(1)
        return _unit_bf16(t * base + (1 - t) * torch.randn(1, D, generator=g) + 0.01 * torch.randn(C, D, generator=g))
    if kind == "equal":
        return _unit_bf16(torch.randn(1, D, generator=g).repeat(C, 1))
    if kind == "dups":
        return _unit_bf16(torch.randn((C + 39) // 40, D, generator=g)).repeat_interleave(40, 0)[:C].contiguous()
    if kind == "zeros":
        w = torch.zeros(C, D)
        w[::97] = torch.randn(len(range(0, C, 97)), D, generator=g)
        return _unit_bf16(w)
    raise ValueError(kind)


def hostile_queries(w, B, kind, seed=11):
    """Image features that land in the hostile region of the bank (near a leaf / near the end); `w` on the device."""
    g = torch.Generator(device=w.device).manual_seed(seed)
    C, D = w.shape
    if kind == "ascending":
        x = w[-1:].float() + 0.02 * torch.randn(B, D, device=w.device, generator=g)
    elif kind == "clustered":
        pick = torch.randint(0, C, (B,), device=w.device, generator=g)
        x = w[pick].float() + 0.3 * torch.randn(B, D, device=w.device, generator=g) / D ** 0.5
    else:
        x = torch.randn(B, D, device=w.device, generator=g)
    return _unit_bf16(x)
