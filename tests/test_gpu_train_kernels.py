"""Element-wise tests of the OM training step's kernels -- the fused masked CE, ``om_backward`` and the dense store
epilogue its two GEMMs run on -- and of the two bank builders, each against a float64 reference computed from the SAME
inputs the kernel receives (bf16 unit rows, fp32 norms, fp32 logits).  The only difference allowed is the kernel's own
rounding, bounded per element; each test says where its bound comes from.  A global ``|a - b|_F / |b|_F`` measure is
not enough here: a lost row of ``d_text`` or a dropped K block moves it by about 1e-2 or less at the cfg-3 head shape.

``test_om_backward_bound_flags_broken_numerics`` needs no GPU: it checks the om_backward bound itself against a CPU
emulation of the kernel's numerics and against two broken variants of it."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from hgrnet_b200 import _cabi, ops
from hgrnet_b200._cabi import HgrError

DEV = "cuda:0"
gpu = pytest.mark.gpu
SCALE = 14.285714                 # exp(logit_scale) at its initial value log(1 / 0.07)


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return _cabi.load()


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _nan_fill(t):
    """Every byte 0xFF: NaN in fp32 and bf16."""
    t.view(torch.uint8).fill_(255)
    return t


def _pad8(v):
    return (v + 7) // 8 * 8


# --------------------------------------------------------------------------- float64 references
def _unit_bf16(n, D, seed):
    """bf16 unit rows and the fp32 norms of the raw rows (what hgr_aggregate_normalize hands the training step);
    the norms differ from row to row."""
    g = _gen(seed)
    raw = torch.randn(n, D, generator=g) * (0.5 + 2.0 * torch.rand(n, 1, generator=g))
    norm = raw.norm(dim=1)
    return (raw / norm[:, None]).to(torch.bfloat16), norm.float()


def _sets(U, T, n, rng):
    """T sets of n distinct columns of [0, U) that together cover every column when T * n >= U (the union of a
    training step is exactly its sampled classes)."""
    order = rng.permutation(U)
    sets = []
    for t in range(T):
        own = order[t * n:(t + 1) * n]
        rest = np.setdiff1d(np.arange(U), own)
        s = np.concatenate([own, rng.choice(rest, n - len(own), replace=False)])
        rng.shuffle(s)
        sets.append(s.astype(np.int32))
    return sets


def _ce_ref(logits, sets, label_pos, weight):
    """float64 masked CE over the T sets (clip_tree.py:275-276, summed over the iterations):
    loss[t] = w_t * mean_b(lse_t(b) - logit(b, label_t)), dl = sum_t w_t / B * (softmax_t - onehot_t), zero outside
    every set.  Also returns mag = sum_t w_t / B * (softmax_t + onehot_t), the scale of each dl element's rounding."""
    lg = logits.double()
    B, U = lg.shape
    loss = torch.zeros(len(sets), dtype=torch.float64)
    dl = torch.zeros(B, U, dtype=torch.float64)
    mag = torch.zeros(B, U, dtype=torch.float64)
    for t, (cols, lp, w) in enumerate(zip(sets, label_pos, weight)):
        cols = torch.as_tensor(np.asarray(cols), dtype=torch.long)
        sub = lg[:, cols]
        lse = torch.logsumexp(sub, dim=1)
        loss[t] = float(w) * (lse - sub[:, lp]).mean()
        p = torch.exp(sub - lse[:, None])
        onehot = torch.zeros_like(p)
        onehot[:, lp] = 1.0
        dl[:, cols] += float(w) / B * (p - onehot)
        mag[:, cols] += float(w) / B * (p + onehot)
    return loss, dl, mag


def _om_ref(dl, lg, x, xn, tn, tnn, s):
    """float64 om_backward on the kernel's inputs and its per-element bound.

    gx = s dl @ tn, gt = s dl^T @ x, then g <- (g - y (y . g)) / n with y the bf16 rows as given; the d_log_scale
    reference is sum(dl * logits).  The kernel's one deliberate loss is rounding dl to bf16: 8 significant bits, so up
    to 2^-8 relative.  The GEMM then sums K exact bf16 products in fp32 (<= K 2^-24 of the absolute sum, K = the padded
    U for d_img, the padded B for d_text) and applies the scale (2^-24); that fp32 part is doubled.  Every element of a
    GEMM output is thus within E1 = (2^-8 + (K + 2) 2^-23) s |dl| @ |tn| (|dl|^T @ |x| for d_text).  The
    normalise-backward is linear in g, so that error reaches the output as at most (E1 + |y| (|y| . E1)) / n.  The
    normalise-backward's own fp32 work adds to it: each lane sums at most D/32 + 4 products y_j g_j with fmaf and a
    5-level shuffle adds them up, <= (D/32 + 9) 2^-24 |y| . |g|; then y_i * dot, the subtraction, 1 / n and the product
    round 4 times, <= 4 2^-24 (|g_i| + |y_i| (|y| . |g|)).  With |g| <= M = (1 + 2^-7) s |dl| @ |tn| (bf16 rounding
    and accumulation included) and doubled, that is Efp = 2^-23 ((D/32 + 13) |y| (|y| . M) + 4 M) / n.  A row whose M is
    zero (an all-zero column of dl) must come out exactly zero."""
    dl, lg, x, tn = dl.double(), lg.double(), x.double(), tn.double()
    B, U = dl.shape
    D = x.shape[1]

    def nb(g, y, n):
        return (g - y * (y * g).sum(1, keepdim=True)) / n.double()[:, None]

    def bound(mag, u, y, n):
        ya = y.abs()
        e1 = u * mag
        m = (1 + 2.0 ** -7) * mag
        efp = 2.0 ** -23 * ((D / 32 + 13) * ya * (ya * m).sum(1, keepdim=True) + 4 * m)
        return (e1 + ya * (ya * e1).sum(1, keepdim=True) + efp) / n.double()[:, None]

    ri, rt = nb(s * dl @ tn, x, xn), nb(s * dl.T @ x, tn, tnn)
    ui, ut = 2.0 ** -8 + (_pad8(U) + 2) * 2.0 ** -23, 2.0 ** -8 + (_pad8(B) + 2) * 2.0 ** -23
    bi = bound(s * dl.abs() @ tn.abs(), ui, x, xn)
    bt = bound(s * dl.abs().T @ x.abs(), ut, tn, tnn)
    return ri, rt, bi, bt, float((dl * lg).sum()), float((dl * lg).abs().sum())


def _om_inputs(B, U, D, seed, ce=False):
    """Inputs of one om_backward call.  dl is the float64 masked CE of 17 sets of 257 classes (rounded to fp32, as the
    kernel writes it) when ``ce``, else Gaussian.  Either way every 7th column from column 3 on is zeroed, except the
    last column, whose packing is the edge of the padded operand."""
    x, xn = _unit_bf16(B, D, seed)
    tn, tnn = _unit_bf16(U, D, seed + 1)
    lg = SCALE * (x.float() @ tn.float().T)
    if ce:
        rng = np.random.RandomState(seed)
        T, n = 17, min(U, 257)
        weight = (rng.rand(T) + 0.05).astype(np.float32)
        dl = _ce_ref(lg, _sets(U, T, n, rng), rng.randint(0, n, size=T), weight)[1].float()
    else:
        dl = torch.randn(B, U, generator=_gen(seed + 2)) * 1e-3
    dl[:, 3:U - 1:7] = 0.0
    return dict(dl=dl, lg=lg, x=x, xn=xn, tn=tn, tnn=tnn)


def _flagged(got, ref, bnd):
    return int(((got.double().cpu() - ref).abs() > bnd).sum())


def _worst(got, ref, bnd):
    """Largest error / bound (an exact zero where the bound is zero counts as 0)."""
    err = (got.double().cpu() - ref).abs()
    return float(torch.where(err == 0, torch.zeros_like(err), err / bnd).max())


def _check_grad(got, ref, bnd, what):
    """Every element within its bound, every row within 1e-2 relative, zero reference rows exactly zero."""
    got = got.double().cpu()
    assert torch.isfinite(got).all(), what + ": non-finite output"
    err = (got - ref).abs()
    bad = int((err > bnd).sum())
    assert bad == 0, "%s: %d elements outside the bound (worst error / bound %.3g)" % (what, bad, _worst(got, ref, bnd))
    rn = ref.norm(dim=1)
    zero = rn == 0
    assert (got[zero] == 0).all(), what + ": rows with a zero reference are not zero"
    if (~zero).any():
        rel = (got - ref).norm(dim=1)[~zero] / rn[~zero]
        assert float(rel.max()) <= 1e-2, "%s: row %d off by %.3g relative" % (what, int(rel.argmax()), float(rel.max()))


def _d_log_scale_tol(B, U, absum):
    """fp32 sum of B*U products: 4 per thread, 5 shuffle levels, 8 warps, then one atomicAdd per 32 x 32 tile of the
    padded extents (any order): at most that many roundings of 2^-24 of the sum of absolute products; doubled."""
    n_add = 4 + 5 + 8 + 1 + (_pad8(U) + 31) // 32 * ((_pad8(B) + 31) // 32)
    return 2 * n_add * 2.0 ** -24 * absum + 1e-30


def _check_om(inp, d_img, d_text):
    ri, rt, bi, bt, _, _ = _om_ref(inp["dl"], inp["lg"], inp["x"], inp["xn"], inp["tn"], inp["tnn"], SCALE)
    _check_grad(d_img, ri, bi, "d_img")
    _check_grad(d_text, rt, bt, "d_text")


def _om_ops(inp, d_ls=None):
    t = {k: v.to(DEV) for k, v in inp.items()}
    return ops.om_backward(t["dl"], t["lg"], t["x"], t["xn"], t["tn"], t["tnn"], SCALE, d_ls)


# --------------------------------------------------------------------------- om_backward: the bound itself (CPU)
def test_om_backward_bound_flags_broken_numerics():
    """At the bench's cfg-3 head shape (B = 256, U = 3,000, D = 1,024; dl of 17 sets of 257), a torch emulation of the
    kernel's numerics (dl rounded to bf16, fp32 GEMMs, fp32 normalise-backward) stays inside the bound of `_om_ref`,
    while a lost d_text row and a d_x GEMM that drops its last partial K block (3,000 = 46 * 64 + 56) are flagged."""
    B, U, D = 256, 3000, 1024
    inp = _om_inputs(B, U, D, seed=5, ce=True)
    ri, rt, bi, bt, _, _ = _om_ref(inp["dl"], inp["lg"], inp["x"], inp["xn"], inp["tn"], inp["tnn"], SCALE)
    dl16, x, tn = inp["dl"].bfloat16().float(), inp["x"].float(), inp["tn"].float()

    def nb(g, y, n):
        return (g - y * (y * g).sum(1, keepdim=True)) / n[:, None]

    gi = nb(SCALE * (dl16 @ tn), x, inp["xn"])
    gt = nb(SCALE * (dl16.T @ x), tn, inp["tnn"])
    _check_grad(gi, ri, bi, "emulated d_img")
    _check_grad(gt, rt, bt, "emulated d_text")
    assert _worst(gi, ri, bi) < 0.5 and _worst(gt, rt, bt) < 0.5

    lost = gt.clone()
    norms = rt.norm(dim=1)
    r = int(torch.where(norms > 0, norms, torch.inf).argmin())     # the touched row with the smallest gradient
    lost[r] = 0.0
    assert _flagged(lost, rt, bt) > 0
    with pytest.raises(AssertionError):
        _check_grad(lost, rt, bt, "d_text")

    k = U // 64 * 64
    gi_tail = nb(SCALE * (dl16[:, :k] @ tn[:k]), x, inp["xn"])
    assert _flagged(gi_tail, ri, bi) > 0
    with pytest.raises(AssertionError):
        _check_grad(gi_tail, ri, bi, "d_img")


# --------------------------------------------------------------------------- om_backward on the GPU
@gpu
@pytest.mark.parametrize("D", [8, 64, 520, 2056])
@pytest.mark.parametrize("U", [1, 9, 130, 1000])
@pytest.mark.parametrize("B", [1, 7, 33, 129, 300])
def test_om_backward_edges(lib, B, U, D):
    """B and U not multiples of 8 or 32, one and several row tiles of the d_text GEMM (M = U), D not a multiple of
    64; bound and per-row check of `_om_ref`, d_log_scale within `_d_log_scale_tol`."""
    inp = _om_inputs(B, U, D, seed=B * 131 + U * 7 + D)
    d_ls = torch.zeros(1, device=DEV)
    d_img, d_text = _om_ops(inp, d_ls)
    _check_om(inp, d_img, d_text)
    _, _, _, _, dls, absum = _om_ref(inp["dl"], inp["lg"], inp["x"], inp["xn"], inp["tn"], inp["tnn"], SCALE)
    assert abs(float(d_ls) - dls) <= _d_log_scale_tol(B, U, absum)


@gpu
@pytest.mark.parametrize("B,U,D", [(256, 3000, 1024), (256, 4369, 1024)])
def test_om_backward_bench_shapes(lib, B, U, D):
    """The bench's OM head shapes with a masked-CE dl.  d_log_scale is ACCUMULATED into a non-zero start value, and
    passing None gives bit-identical gradients."""
    inp = _om_inputs(B, U, D, seed=U, ce=True)
    start = 0.75
    d_ls = torch.full((1,), start, device=DEV)
    d_img, d_text = _om_ops(inp, d_ls)
    _check_om(inp, d_img, d_text)
    _, _, _, _, dls, absum = _om_ref(inp["dl"], inp["lg"], inp["x"], inp["xn"], inp["tn"], inp["tnn"], SCALE)
    assert abs(float(d_ls) - (start + dls)) <= _d_log_scale_tol(B, U, absum) + 2.0 ** -24 * start
    d_img2, d_text2 = _om_ops(inp, None)
    assert torch.equal(d_img2, d_img) and torch.equal(d_text2, d_text)


@gpu
@pytest.mark.parametrize("B,U,D", [(33, 130, 520), (129, 1000, 64), (7, 9, 2056)])
def test_om_backward_c_abi_poisoned_buffers(lib, B, U, D):
    """Through the C ABI: workspace, d_img and d_text filled with 0xFF bytes (NaN) before the call, and dlogits /
    logits with ldl = U + 8 whose extra columns hold NaN.  Every output must be finite and within bound -- no unwritten
    padding element of the workspace and no column beyond U is read -- and equal, bit for bit, to a clean call through
    ops; the extra input columns are left alone."""
    inp = _om_inputs(B, U, D, seed=3 * B + U)
    ldl = U + 8
    dl_buf = torch.full((B, ldl), float("nan"))
    lg_buf = torch.full((B, ldl), float("nan"))
    dl_buf[:, :U], lg_buf[:, :U] = inp["dl"], inp["lg"]
    dl_buf, lg_buf = dl_buf.to(DEV), lg_buf.to(DEV)
    x, xn, tn, tnn = (inp[k].to(DEV) for k in ("x", "xn", "tn", "tnn"))
    ws = torch.full((lib.hgr_om_backward_workspace_bytes(B, U, D),), 255, dtype=torch.uint8, device=DEV)
    d_img = _nan_fill(torch.empty(B, D, device=DEV))
    d_text = _nan_fill(torch.empty(U, D, device=DEV))
    d_ls = torch.full((1,), -0.5, device=DEV)
    _cabi.check(lib.hgr_om_backward(dl_buf.data_ptr(), lg_buf.data_ptr(), ldl, B, U, D, x.data_ptr(), xn.data_ptr(),
                                    tn.data_ptr(), tnn.data_ptr(), SCALE, d_img.data_ptr(), d_text.data_ptr(),
                                    d_ls.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()))
    _check_om(inp, d_img, d_text)
    _, _, _, _, dls, absum = _om_ref(inp["dl"], inp["lg"], inp["x"], inp["xn"], inp["tn"], inp["tnn"], SCALE)
    assert abs(float(d_ls) - (dls - 0.5)) <= _d_log_scale_tol(B, U, absum) + 2.0 ** -24
    assert torch.isnan(dl_buf[:, U:]).all() and torch.isnan(lg_buf[:, U:]).all()
    clean_img, clean_text = _om_ops(inp)
    assert torch.equal(d_img, clean_img) and torch.equal(d_text, clean_text)


@gpu
def test_om_backward_reuses_workspace_after_a_larger_call(lib):
    """ops caches one workspace per stream.  A small call after a large one runs on the large call's leftovers in
    the padding of its packed operands, and again on a workspace of 0xFF bytes: same result, within bound."""
    _om_ops(_om_inputs(256, 3000, 1024, seed=11, ce=True))
    key = ("om_bwd", torch.device(DEV).index, ops._stream())
    ws = ops._workspaces[key]
    small = _om_inputs(33, 130, 520, seed=12)
    d_img, d_text = _om_ops(small)
    assert ops._workspaces[key] is ws, "the small call should have reused the cached workspace"
    _check_om(small, d_img, d_text)
    ws.fill_(255)
    d_img2, d_text2 = _om_ops(small)
    assert torch.equal(d_img2, d_img) and torch.equal(d_text2, d_text)


# --------------------------------------------------------------------------- masked CE
def _ce_case(B, U, T, n, seed, amp=3.0, where=None, uniform=False):
    rng = np.random.RandomState(seed)
    g = _gen(seed)
    logits = (torch.rand(B, U, generator=g) * 2 - 1) * amp if uniform else torch.randn(B, U, generator=g) * amp
    sets = _sets(U, T, n, rng)
    if where == "first":
        lps = [0] * T
    elif where == "last":
        lps = [n - 1] * T
    else:
        lps = [int(v) for v in rng.randint(0, n, size=T)]
    weight = (rng.rand(T) + 0.05).astype(np.float32)
    return logits, sets, lps, weight


def _ce_dev(sets, lps, weight):
    set_ptr = np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.int32)
    set_col = np.concatenate(sets).astype(np.int32) if sets else np.zeros(0, np.int32)
    return [torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
            for a in (set_ptr, set_col, np.asarray(lps, np.int32), np.asarray(weight, np.float32))]


def _check_ce(logits, sets, lps, weight, loss, dl):
    """Bounds against the float64 `_ce_ref`, for fp32 evaluation with amax = max |logit|: l - m and l - lse are
    rounded by <= 2^-24 * 2 amax, expf / logf add a few ulps, the block sums of <= 1,025 exponentials <= 16 * 2^-24,
    so lse is within 2^-24 (3 amax + 16) and each softmax entry within 2^-24 (5 amax + 32) relative; the T-term sum
    into a dl element adds T 2^-24 of its magnitude.  Doubled: eps = 2^-24 (8 amax + 64 + 2 T) per unit of
    `mag`, plus 2^-100 absolute for exponentials that underflow in fp32.  The loss adds its batch mean: one warp sums B
    non-negative terms, (B / 32 + 8) 2^-24 relative, also doubled."""
    B = logits.shape[0]
    T = len(sets)
    ref_l, ref_dl, mag = _ce_ref(logits, sets, lps, weight)
    amax = float(logits.abs().max())
    eps = 2.0 ** -24 * (8 * amax + 64 + 2 * T)
    w = torch.as_tensor(np.asarray(weight, np.float64))
    lerr = (loss.double().cpu() - ref_l).abs()
    assert (lerr <= w * eps + 2 * (B / 32 + 8) * 2.0 ** -24 * ref_l.abs()).all(), (loss.cpu(), ref_l)
    if dl is None:
        return
    dl = dl.double().cpu()
    assert torch.isfinite(dl).all()
    assert (dl[mag == 0] == 0).all(), "dlogits not zero outside every set"
    err = (dl - ref_dl).abs()
    bnd = eps * mag + 2.0 ** -100
    assert (err <= bnd).all(), "dlogits: %d elements outside the bound (worst error / bound %.3g)" % (
        int((err > bnd).sum()), float((err / bnd).max()))


def _ce_run(logits, sets, lps, weight):
    args = _ce_dev(sets, lps, weight)
    loss, dl = ops.masked_ce(logits.to(DEV), *args)
    _check_ce(logits, sets, lps, weight, loss, dl)
    loss2, none = ops.masked_ce(logits.to(DEV), *args, need_grad=False)
    assert none is None and torch.equal(loss2, loss)
    return loss, dl


@gpu
def test_masked_ce_cfg3_shape(lib):
    """The bench's cfg-3 head: B = 256, a union of U = 3,000 classes, T = 17 sets of 257."""
    _ce_run(*_ce_case(256, 3000, 17, 257, seed=1))


@gpu
@pytest.mark.parametrize("where", ["first", "last"])
@pytest.mark.parametrize("n", [1, 256, 257, 1025])
def test_masked_ce_set_sizes(lib, n, where):
    """Sets of one class (loss and gradient exactly zero), of one and of just over one 256-thread block, and of 1,025;
    the label at position 0 or n - 1 of its set."""
    logits, sets, lps, weight = _ce_case(33, 2000, 3, n, seed=n, where=where)
    loss, dl = _ce_run(logits, sets, lps, weight)
    if n == 1:
        assert (loss == 0).all() and (dl == 0).all()


@gpu
def test_masked_ce_large_logits_single_row(lib):
    """B = 1 and logits up to magnitude 100 (scale 100): most exponentials of a set underflow in fp32."""
    _ce_run(*_ce_case(1, 700, 5, 257, seed=7, amp=100.0, uniform=True))


@gpu
@pytest.mark.parametrize("U", [20000, 51200])
def test_masked_ce_wide_union(lib, U):
    """Unions whose fp32 row buffer needs more than 48 KB of dynamic shared memory, up to the largest accepted
    (51,200 classes = 200 KB); one class more is refused."""
    _ce_run(*_ce_case(4, U, 3, 1025, seed=U))
    if U == 51200:
        logits, sets, lps, weight = _ce_case(2, U + 1, 1, 4, seed=1)
        with pytest.raises(HgrError):
            ops.masked_ce(logits.to(DEV), *_ce_dev(sets, lps, weight))


@gpu
def test_masked_ce_c_abi_padded_and_poisoned(lib):
    """Through the C ABI with ldl = U + 8: dlogits and the workspace hold NaN before the call and the logits' extra
    columns hold NaN.  Every dlogits element in [0, U) is overwritten (zero outside the sets), the sentinels beyond U
    are untouched."""
    B, U, T, n = 33, 1000, 5, 257
    logits, sets, lps, weight = _ce_case(B, U, T, n, seed=9)
    ldl = U + 8
    lg_buf = torch.full((B, ldl), float("nan"))
    lg_buf[:, :U] = logits
    lg_buf = lg_buf.to(DEV)
    dl_buf = torch.full((B, ldl), 12345.0, device=DEV)
    _nan_fill(dl_buf[:, :U])
    loss = torch.full((T,), float("nan"), device=DEV)
    ws = torch.full((lib.hgr_masked_ce_workspace_bytes(B, U, T),), 255, dtype=torch.uint8, device=DEV)
    sp, sc, lp, w = _ce_dev(sets, lps, weight)
    _cabi.check(lib.hgr_masked_ce(lg_buf.data_ptr(), ldl, B, U, sp.data_ptr(), sc.data_ptr(), lp.data_ptr(), w.data_ptr(),
                                  T, loss.data_ptr(), dl_buf.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()))
    _check_ce(logits, sets, lps, weight, loss, dl_buf[:, :U])
    assert (dl_buf[:, U:] == 12345.0).all()


@gpu
def test_masked_ce_without_sets(lib):
    """T == 0: an empty loss and a gradient that is zero everywhere -- written, not left as it was."""
    B, U = 5, 300
    logits = torch.randn(B, U, generator=_gen(2)).to(DEV)
    loss, dl = ops.masked_ce(logits, *_ce_dev([], [], []))
    assert loss.shape == (0,) and dl.shape == (B, U) and (dl == 0).all()
    loss, none = ops.masked_ce(logits, *_ce_dev([], [], []), need_grad=False)
    assert loss.shape == (0,) and none is None
    ldl = U + 8
    lg_buf = torch.zeros(B, ldl, device=DEV)
    lg_buf[:, :U] = logits
    dl_buf = torch.full((B, ldl), 12345.0, device=DEV)
    _nan_fill(dl_buf[:, :U])
    ws = torch.full((lib.hgr_masked_ce_workspace_bytes(B, U, 0),), 255, dtype=torch.uint8, device=DEV)
    _cabi.check(lib.hgr_masked_ce(lg_buf.data_ptr(), ldl, B, U, None, None, None, None, 0, None, dl_buf.data_ptr(),
                                  ws.data_ptr(), ws.numel(), ops._stream()))
    assert (dl_buf[:, :U] == 0).all() and (dl_buf[:, U:] == 12345.0).all()


# --------------------------------------------------------------------------- dense store epilogue: out= arguments
@gpu
@pytest.mark.parametrize("impl", ["simt", "tcgen05"])
@pytest.mark.parametrize("B,C,D", [(37, 313, 64), (3000, 1024, 256)])
def test_logits_dense_into_column_slice(lib, impl, B, C, D):
    """``out`` as a column slice of a wider fp32 buffer (ldo = C + 40 > C): the slice gets exactly what a dense
    output gets, every cell around it keeps its sentinel."""
    imp = {"simt": ops.HGR_IMPL_SIMT, "tcgen05": ops.HGR_IMPL_TCGEN05}[impl]
    x, _ = _unit_bf16(B, D, 1)
    w, _ = _unit_bf16(C, D, 2)
    x, w = x.to(DEV), w.to(DEV)
    want = ops.logits_dense(x, w, scale=SCALE, impl=imp)
    buf = torch.full((B, C + 40), -777.0, device=DEV)
    out = buf[:, 8:8 + C]
    assert out.stride(0) == C + 40
    got = ops.logits_dense(x, w, scale=SCALE, impl=imp, out=out)
    assert got.data_ptr() == out.data_ptr()
    assert torch.equal(out, want)
    assert (buf[:, :8] == -777.0).all() and (buf[:, 8 + C:] == -777.0).all()
    # one row: any row stride is fine (here a transposed column, stride(0) == 1)
    col = torch.full((C + 8, 1), -777.0, device=DEV)
    one = col[4:4 + C].t()
    assert one.shape == (1, C) and one.stride() == (1, 1)
    ops.logits_dense(x[:1], w, scale=SCALE, impl=imp, out=one)
    assert torch.equal(one, want[:1])
    assert (col[:4] == -777.0).all() and (col[4 + C:] == -777.0).all()


@gpu
def test_logits_dense_rejects_bad_out_before_launch(lib):
    """An ``out`` of the wrong dtype, shape, layout or device raises before the library is called: nothing is
    launched and the tensor is unchanged.  (Without the check a bf16 [B, C] out received fp32 stores: twice its
    size.)  The cases are ordered so that each one that got through would still write inside its own buffer until
    the bf16 one."""
    B, C, D = 64, 200, 128
    x, _ = _unit_bf16(B, D, 1)
    w, _ = _unit_bf16(C, D, 2)
    x, w = x.to(DEV), w.to(DEV)
    wide = torch.zeros(B, 2 * C, device=DEV)
    bad = [torch.zeros(B, C + 1, device=DEV),                      # shape
           torch.zeros(1, C, device=DEV).expand(B, C),             # stride(0) == 0: rows on top of each other
           wide[:, ::2],                                           # stride(1) == 2
           torch.zeros(C, B, device=DEV).t(),                      # column-major
           torch.zeros(B, C, dtype=torch.float64, device=DEV),     # dtype
           torch.zeros(B, C),                                      # host memory
           torch.zeros(B, C, dtype=torch.bfloat16, device=DEV)]    # dtype, and half the bytes
    torch.cuda.synchronize()
    for out in bad:
        before = out.clone()
        n0 = _cabi.launch_count()
        with pytest.raises(ValueError, match="out must be"):
            ops.logits_dense(x, w, out=out)
        assert _cabi.launch_count() == n0
        assert torch.equal(out, before)
    assert (wide == 0).all()


# --------------------------------------------------------------------------- bank builders
@gpu
@pytest.mark.parametrize("D", [8, 520, 1024])
@pytest.mark.parametrize("n", [1, 37, 4096 + 5])
@pytest.mark.parametrize("in_dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_normalize_rows_dual(lib, in_dtype, n, D):
    """The production bank refresh: ``out`` equals ``normalize_rows`` bit for bit and the float64 normalised rows
    within bf16 rounding (2^-8 relative) plus the fp32 norm (<= (D + 4) 2^-24 relative); every row with
    dst_map >= 0 -- the chunk's last row among them -- is copied to ``out2[dst_map[r]]``, and the rows of ``out2``
    that nothing maps to keep their sentinel."""
    g = _gen(n + D)
    E = (torch.randn(n, D, generator=g) * (0.3 + torch.rand(n, 1, generator=g))).to(in_dtype)
    rng = np.random.RandomState(n + D)
    mapped = rng.rand(n) < 0.6
    mapped[-1] = True
    n2 = int(mapped.sum()) + 5
    dst = np.full(n, -1, np.int32)
    dst[mapped] = rng.permutation(n2)[:int(mapped.sum())]
    sentinel = -7.0
    out = torch.full((n, D), sentinel, dtype=torch.bfloat16, device=DEV)
    out2 = torch.full((n2, D), sentinel, dtype=torch.bfloat16, device=DEV)
    Ed = E.to(DEV)
    ops.normalize_rows_dual(Ed, out, torch.from_numpy(dst).to(DEV), out2)
    assert torch.equal(out, ops.normalize_rows(Ed))
    ref = E.double() / E.double().norm(dim=1, keepdim=True)
    assert ((out.cpu().double() - ref).abs() <= (2.0 ** -8 + (D + 4) * 2.0 ** -24) * ref.abs()).all()
    m = torch.from_numpy(mapped)
    o2 = out2.cpu()
    assert torch.equal(o2[torch.from_numpy(dst[mapped]).long()], out.cpu()[m])
    unmapped = np.setdiff1d(np.arange(n2), dst[mapped])
    assert len(unmapped) == 5 and (o2[torch.from_numpy(unmapped).long()] == sentinel).all()
    alone = torch.full((n, D), sentinel, dtype=torch.bfloat16, device=DEV)
    ops.normalize_rows_dual(Ed, alone)
    assert torch.equal(alone, out)


@gpu
def test_normalize_rows_dual_limits(lib):
    """D = 1,032 is refused (the kernel holds at most 1,024 elements of a row); n = 0 launches nothing."""
    E = torch.randn(4, 1032, device=DEV)
    with pytest.raises(HgrError):
        ops.normalize_rows_dual(E, torch.empty(4, 1032, dtype=torch.bfloat16, device=DEV))
    out2 = torch.full((3, 64), 1.0, dtype=torch.bfloat16, device=DEV)
    n0 = _cabi.launch_count()
    ops.normalize_rows_dual(torch.empty(0, 64, device=DEV), torch.empty(0, 64, dtype=torch.bfloat16, device=DEV),
                            torch.empty(0, dtype=torch.int32, device=DEV), out2)
    assert _cabi.launch_count() == n0 and (out2 == 1.0).all()


ROW_LENS = [1, 31, 32, 33, 63, 64, 65, 300]


@gpu
@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("D", [8, 520, 2048, 2056, 4096])
def test_aggregate_csr_long_rows(lib, D, weighted):
    """CSR rows of 1 to 300 entries: around each 32-entry reload of the column ids / weights, with and without
    weights.  D = 8 / 520 / 2,048 run the register kernel with 1 / 3 / 8 vectors per lane, 2,056 and 4,096 the generic
    kernel.  Against float64: the fp32 sum of a row's n terms is within n 2^-24 m (m = sum |w_j| |E[c_j]| per element),
    which moves the normalised element by <= n 2^-24 (m_i + |ref_i| |m|) / |acc|; the fp32 norm and division add
    (D + 4) 2^-24 |ref_i|.  Both doubled."""
    n_src = 500
    E = torch.randn(n_src, D, generator=_gen(D))
    rng = np.random.RandomState(D + weighted)
    lens = np.asarray(ROW_LENS * 2)
    rng.shuffle(lens)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rng.randint(0, n_src, size=int(rowptr[-1])).astype(np.int32)
    w = (rng.rand(int(rowptr[-1])) + 0.1).astype(np.float32)
    t = lambda a: torch.from_numpy(a).to(DEV)
    got, norm = ops.aggregate_normalize(E.to(DEV), t(rowptr), t(col), t(w) if weighted else None,
                                        out_dtype=torch.float32, return_norm=True)
    wj = torch.from_numpy(w).double() if weighted else torch.ones(len(col), dtype=torch.float64)
    rows = torch.repeat_interleave(torch.arange(len(lens)), torch.from_numpy(lens))
    src = E.double()[torch.from_numpy(col).long()]
    acc = torch.zeros(len(lens), D, dtype=torch.float64).index_add_(0, rows, wj[:, None] * src)
    mag = torch.zeros(len(lens), D, dtype=torch.float64).index_add_(0, rows, wj[:, None].abs() * src.abs())
    an = acc.norm(dim=1, keepdim=True)
    ref = acc / an
    n = torch.from_numpy(lens).double()[:, None]
    bnd = 2 * (n * 2.0 ** -24 * (mag + ref.abs() * mag.norm(dim=1, keepdim=True)) / an + (D + 4) * 2.0 ** -24 * ref.abs())
    err = (got.cpu().double() - ref).abs()
    assert (err <= bnd).all(), "%d elements outside the bound (worst error / bound %.3g)" % (
        int((err > bnd).sum()), float((err / bnd).max()))
    nb = 2 * (n[:, 0] * 2.0 ** -24 * mag.norm(dim=1) + (D + 4) * 2.0 ** -24 * an[:, 0])
    assert ((norm.cpu().double() - an[:, 0]).abs() <= nb).all()
