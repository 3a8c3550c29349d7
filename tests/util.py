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


def order_key(v):
    """int64 restatement of ``topk_list.cuh::order_key``: a larger key is a larger value, and -0 sorts below +0."""
    b = v.float().contiguous().view(torch.int32).long() & 0xFFFFFFFF
    return torch.where(b >= 0x80000000, b ^ 0xFFFFFFFF, b | 0x80000000)


def _ids_of_rows(rows, col_id, id_base):
    rows = rows.long()
    ids = col_id.long()[rows.clamp_min(0)] if col_id is not None else rows + id_base
    return torch.where(rows >= 0, ids, torch.full_like(ids, -1)).int()


def reference_topk(X, bank, K, scale=1.0, col_id=None, id_base=0):
    """Bit-exact reference of every tcgen05 top-K epilogue: a sort of the dense logits of the same GEMM.

    ``ops.logits_dense`` (tcgen05) holds the fp32 accumulators each epilogue sees -- their rounding does not depend on
    the element's place in the tile.  Rows are ordered by (value desc, bank row asc), the value compared through the
    kernels' order key (a stable descending sort of that key).  The ORDER comes from the unscaled accumulators and the
    VALUES from ``logits_dense(scale=s)``: the lists are sorted before the merge multiplies by ``scale``, so where two
    distinct accumulators round to the same scaled value the kernels keep the unscaled order, and so does this.
    Returns device ``(val [B, K] fp32, idx [B, K] int32 ids)``, padded with (-inf, -1) when C < K."""
    from hgrnet_b200 import ops
    B, C = X.shape[0], bank.shape[0]
    acc = ops.logits_dense(X, bank, scale=1.0, impl=ops.HGR_IMPL_TCGEN05)
    scaled = acc if scale == 1.0 else ops.logits_dense(X, bank, scale=scale, impl=ops.HGR_IMPL_TCGEN05)
    Kv = min(K, C)
    rows = torch.sort(order_key(acc), dim=1, descending=True, stable=True).indices[:, :Kv]
    val = torch.full((B, K), float("-inf"), device=X.device)
    idx = torch.full((B, K), -1, dtype=torch.int32, device=X.device)
    val[:, :Kv] = scaled.gather(1, rows)
    idx[:, :Kv] = _ids_of_rows(rows, None if col_id is None else col_id.to(X.device), id_base)
    return val, idx


def reference_hits(idx, targets):
    """Hit@{1,2,5,10,20} the kernels count for lists ``idx``: a target below 0 (padding) is never a hit, also not
    against the -1 that pads a list when C < K."""
    t = torch.as_tensor(targets).long().cpu()
    return hits_from_idx(idx, torch.where(t < 0, torch.full_like(t, -2), t))


def check_topk_f64(val, idx, X, bank, K, scale=1.0, col_id=None, id_base=0, rows=None):
    """Float64-certified check of top-K lists whose sums are not the tensor core's (``simt``, rows the production
    kernel repaired on the CUDA cores).  R = float64 logits (exact products of the bf16 inputs), E = (D + 2) 2^-23
    scale |x| @ |w| the bound of an fp32 sum of D products and the scaling.  Per row: every value is within E of
    scale * R of its bank row; values do not increase, ids are distinct, the padding (-inf, -1) appears exactly when
    C < K; and no bank row left out has scale * R - E above the K-th value.  ``rows``: the rows to check (all)."""
    B, D = X.shape
    C = bank.shape[0]
    dev = X.device
    sel = torch.arange(B, device=dev) if rows is None else torch.as_tensor(rows, device=dev).long()
    if sel.numel() == 0:
        return
    x, w = X[sel].double(), bank.double()
    R = scale * (x @ w.T)
    E = (D + 2) * 2.0 ** -23 * scale * (x.abs() @ w.abs().T)
    v, ids = val.to(dev)[sel].double(), idx.to(dev)[sel].long()
    Kv = min(K, C)
    if Kv < K:
        assert torch.isinf(v[:, Kv:]).all() and (v[:, Kv:] < 0).all() and (ids[:, Kv:] == -1).all(), "padding"
    v, ids = v[:, :Kv], ids[:, :Kv]
    assert (ids >= 0).all(), "a list of C >= K columns holds an empty entry"
    if col_id is not None:
        row_of = torch.full((int(col_id.max()) + 1,), -1, dtype=torch.long, device=dev)
        row_of[col_id.to(dev).long()] = torch.arange(C, device=dev)
        r = row_of[ids]
    else:
        r = ids - id_base
    assert ((r >= 0) & (r < C)).all(), "an id names no bank row"
    assert (r.sort(1).values[:, 1:] != r.sort(1).values[:, :-1]).all(), "an id appears twice in a row"
    assert (v[:, :-1] >= v[:, 1:]).all(), "values not sorted descending"
    err = (v - R.gather(1, r)).abs() - E.gather(1, r)
    assert (err <= 0).all(), "value off its float64 logit by more than the bound: %g" % float(err.max())
    left = torch.ones_like(R, dtype=torch.bool).scatter_(1, r, False)
    beat = left & ((R - E) > v[:, -1:])
    assert not beat.any(), "row %d: bank rows left out beat the K-th value" % int(sel[beat.any(1)][0])


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
