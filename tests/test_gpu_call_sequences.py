"""No kernel's result may depend on what an earlier call left behind.

Several kernels keep state in memory that outlives a call, so that a batch needs no memset and a call can be captured
in a graph: the per-stream scoring workspace (``ops._workspace``: the header words ``stats[0]`` = rows the merge
re-scanned, ``stats[1]`` = the floor sketch's epoch, ``stats[2]`` = its finished CTAs, then the partial lists or the
sketch's ``[B][20]`` floor words, which are never cleared), the per-level arg-max words of TOR / POR (``_hier_workspace``,
handed back zeroed by the finishing or push kernel), the host-side plan cache of the grouped schedule, and the counters
every metric kernel increments.

Every test here runs calls in sequence on one stream, chosen so that stale state is LARGER than anything the next call
produces: batch A puts its queries at cluster centres of a clustered bank (at least K logits per row near 1), batch B
is anti-aligned with those centres or random (nothing above 0.5).  Every call's outputs start poisoned, and every call
must equal a reference computed for that call alone: exact and sketch lists ``reference_topk`` bit for bit, hits
included; production lists the ``_check`` rule of ``test_gpu_topk_exact``; ``simt`` the float64 check."""
from __future__ import annotations

import pytest
import torch

import tests.test_gpu_topk_exact as exact_tests
from tests.test_gpu_topk_exact import _check, _impl, _poisoned, _rand
from tests.util import _unit_bf16, check_topk_f64, hostile_bank, reference_hits, reference_topk

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
K = 20

# cfg 2, and a ragged shape whose floor region ([B][20] words) and partial lists overlap the workspace differently
SHAPES = [(512, 21841, 1024), (257, 4097, 1032)]
WRITERS = ("simt", "tcgen05_exact", "tcgen05", "tcgen05_sketch", "share2", "share4", "splits", "scatter",
           "scatter_bounded", "masked_ce", "om_backward", "logits_dense")
READERS = ("tcgen05_sketch", "tcgen05_exact", "tcgen05", "simt")

ops = None


@pytest.fixture(scope="module", autouse=True)
def _load():
    global ops
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from hgrnet_b200 import ops as _ops
    ops = _ops
    exact_tests.ops = _ops          # _check reads the module global of its own file
    yield
    torch.cuda.synchronize()


def _hot(bank, B, seed):
    """Queries at the centres of full 64-row clusters of ``hostile_bank(kind="clustered")``: every row has its 64
    siblings near cosine 1."""
    g = torch.Generator().manual_seed(seed)
    C = bank.shape[0]
    c = torch.randint(0, C // 64, (B,), generator=g)
    centres = bank[:C // 64 * 64].float().view(C // 64, 64, -1).mean(1)
    return _unit_bf16(centres[c.to(bank.device)] + 0.01 * torch.randn(B, centres.shape[1], generator=g).to(bank.device))


def _cold(bank, B, seed):
    """Even rows anti-aligned with a cluster centre, odd rows random directions: no logit near the hot ones."""
    g = torch.Generator().manual_seed(seed)
    x = -_hot(bank, B, seed).float()
    x[1::2] = torch.randn(x[1::2].shape, generator=g).to(bank.device)
    return _unit_bf16(x)


def _targets(ref_i, seed):
    """Ids at varying ranks of each row's reference list (hits at every cut), with padding rows (-1)."""
    B = ref_i.shape[0]
    r = torch.randint(0, 2 * K, (B,), generator=torch.Generator().manual_seed(seed)).to(ref_i.device)
    t = torch.where(r < K, ref_i.gather(1, r.clamp_max(K - 1)[:, None]).squeeze(1), torch.full_like(r, 10 ** 6).int())
    t[::7] = -1
    return t.int()


_CASES = {}


def _case(B, C, D):
    """Bank, batches A / B / W (W: the writers' unrelated hot batch), their references and targets; built once."""
    key = (B, C, D)
    if key not in _CASES:
        bank = hostile_bank(C, D, "clustered", seed=C).to(DEV)
        c = dict(bank=bank, X={"A": _hot(bank, B, 1), "B": _cold(bank, B, 2), "W": _hot(bank, B, 3)})
        c["ref"] = {k: reference_topk(x, bank, K) for k, x in c["X"].items()}
        c["t"] = {k: _targets(r[1], i) for i, (k, r) in enumerate(c["ref"].items())}
        # the adversarial order: every stale value of A (or W) is above everything B produces
        assert float(c["ref"]["A"][0][:, K - 1].min()) > 0.5 and float(c["ref"]["W"][0][:, K - 1].min()) > 0.5
        assert float(c["ref"]["B"][0].max()) < 0.5
        _CASES[key] = c
    return _CASES[key]


def _write(name, X, bank):
    """One call of ``name`` on unrelated inputs; returns what must stay alive until the stream has run it."""
    B, D = X.shape
    C = bank.shape[0]
    if name in ("simt", "tcgen05_exact", "tcgen05", "tcgen05_sketch"):
        return ops.score_topk(X, bank, K=K, impl=_impl(name))
    if name.startswith("share"):
        return ops.score_topk(X, bank, K=K, grid_share=int(name[-1]))
    if name == "splits":
        return ops.score_topk_splits(X, bank, [C // 3, C], [1, 3], 2, K=K)
    if name in ("scatter", "scatter_bounded"):
        v, i, b = _poisoned(B, K) + (torch.empty(B, device=DEV),)
        bounded = name == "scatter_bounded"
        ops.score_topk_scatter(X, bank, [v.data_ptr()], [i.data_ptr()], B, K=K,
                               bound_block_ptrs=[b.data_ptr()] if bounded else None, C_total=4 * C if bounded else 0)
        return v, i, b
    if name == "masked_ce":
        g = torch.Generator(device=DEV).manual_seed(5)
        logits = 10 * torch.randn(B, 64, device=DEV, generator=g)
        sets = torch.tensor([0, 20, 40, 64], dtype=torch.int32, device=DEV)
        return ops.masked_ce(logits, sets, torch.arange(64, dtype=torch.int32, device=DEV),
                             torch.tensor([0, 1, 2], dtype=torch.int32, device=DEV), torch.ones(3, device=DEV))
    if name == "om_backward":
        U = 64
        g = torch.Generator(device=DEV).manual_seed(6)
        dl, lg = 1e-3 * torch.randn(B, U, device=DEV, generator=g), torch.randn(B, U, device=DEV, generator=g)
        return ops.om_backward(dl, lg, X, torch.ones(B, device=DEV), bank[:U].contiguous(), torch.ones(U, device=DEV), 1.0)
    if name == "logits_dense":
        return ops.logits_dense(X, bank)
    raise ValueError(name)


def _read_and_check(impl, case, which):
    """``impl`` on batch ``which`` into poisoned outputs: lists and hits against that batch's own reference."""
    X, bank = case["X"][which], case["bank"]
    ref_v, ref_i = case["ref"][which]
    t = case["t"][which]
    hits = ops.new_hits(DEV)
    val, idx = ops.score_topk(X, bank, targets=t, K=K, hits=hits, impl=_impl(impl), out=_poisoned(X.shape[0], K))
    _check(impl, val, idx, ref_v, ref_i, X, bank, K, 1.0)
    assert hits.tolist() == reference_hits(idx, t), (impl, which)
    if impl in ("tcgen05_exact", "tcgen05_sketch"):
        assert hits.tolist() == reference_hits(ref_i, t), (impl, which)


# ---- 1. the shared scoring workspace -----------------------------------------------------------------------------

@pytest.mark.parametrize("writer", WRITERS)
@pytest.mark.parametrize("B,C,D", SHAPES)
def test_reader_after_writer_on_two_batches(B, C, D, writer):
    """On one stream: ``writer`` on an unrelated hot batch, then each reader on A, then on B.  A sketch whose epoch
    stopped advancing filters B against A's floors and loses B's top-K; a header overwritten by a caller outside the
    scoring family does that, or breaks the re-scan count the production check relies on."""
    case = _case(B, C, D)
    for reader in READERS:
        keep = _write(writer, case["X"]["W"], case["bank"])
        for which in ("A", "B"):
            try:
                _read_and_check(reader, case, which)
            except AssertionError as e:
                raise AssertionError("%s -> %s on batch %s: %s" % (writer, reader, which, e)) from None
        del keep


# three different batches at shapes whose sketch grids differ (gridDim.x changes between launches); the first shape is
# the largest, so that the stream's workspace is not reallocated (a new one starts zeroed and would hide stale words)
_SKETCH_SEQ = [((512, 21841, 1024), "A"), ((257, 4097, 1032), "B"), ((129, 300, 1032), "B"), ((512, 21841, 1024), "B")]


def test_sketch_sequence_on_changing_grids():
    for (B, C, D), which in _SKETCH_SEQ:
        _read_and_check("tcgen05_sketch", _case(B, C, D), which)


def test_sketch_sequence_replayed_from_graphs():
    """The benchmark's pattern: four query buffers, one captured sketch call per buffer, replayed in turn with hot
    and cold batches; every replay's lists are those of its own buffer."""
    case = _case(*SHAPES[0])
    bank = case["bank"]
    qs = [case["X"][w].clone() for w in ("A", "B", "W", "B")]
    outs = [_poisoned(SHAPES[0][0], K) for _ in qs]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    graphs = []
    with torch.cuda.stream(st):
        ops.score_topk(qs[0], bank, K=K, impl=ops.HGR_IMPL_TCGEN05_SKETCH)      # warm-up: this stream's workspace
        for q, out in zip(qs, outs):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                ops.score_topk(q, bank, K=K, impl=ops.HGR_IMPL_TCGEN05_SKETCH, out=out)
            graphs.append(g)
        for rep in range(2):
            for i, (g, w) in enumerate(zip(graphs, ("A", "B", "W", "B"))):
                for o in outs[i]:
                    o.fill_(float("nan") if o.dtype == torch.float32 else 0x7FFFFFFF)
                g.replay()
                st.synchronize()
                ref_v, ref_i = case["ref"][w]
                bad = ~((outs[i][0] == ref_v).all(1) & (outs[i][1] == ref_i).all(1))
                assert not bad.any(), "replay %d of graph %d (batch %s): %d rows differ, first %d" % (
                    rep, i, w, int(bad.sum()), int(bad.nonzero()[0]))
    torch.cuda.synchronize()


def test_rescan_count_is_the_last_scoring_call():
    """``last_rescan_count()`` after a production call that repairs rows, after callers outside the scoring family
    (which must leave it alone), and after a production call that repairs none (which must read 0)."""
    B, C, D, Kr = 129, 300, 64, 12
    plan = ops.score_topk_plan(B, C, D, Kr)
    assert plan["list_len"] < Kr and ops.score_topk_plan(B, C, D, 8)["list_len"] >= 8
    cpw = plan["cols_per_worker"]
    g = torch.Generator().manual_seed(7)
    X = _unit_bf16(torch.randn(1, D, generator=g) + 0.5 * torch.randn(B, D, generator=g) / D ** 0.5).to(DEV)
    bank = _rand(C, D, 8).clone()
    mean = X.float().mean(0)
    mean = mean / mean.norm()
    r0 = (C // 2) // cpw * cpw
    n = min(cpw, 40)
    bank[r0:r0 + n] = _unit_bf16(3 * mean[None, :].cpu() + torch.randn(n, D, generator=g) / D ** 0.5).to(DEV)
    ops.score_topk(X, bank, K=32)                    # sizes the stream's workspace for everything below
    val, idx = ops.score_topk(X, bank, K=Kr)
    repaired = ops.last_rescan_count(DEV)
    assert repaired > 0, "the adversarial bank should overflow speculative lists"
    ref = reference_topk(X, bank, Kr)
    _check("tcgen05", val, idx, *ref, X, bank, Kr, 1.0)
    for writer in ("simt", "masked_ce", "om_backward", "logits_dense"):
        keep = _write(writer, X, bank)
        assert ops.last_rescan_count(DEV) == repaired, writer
        del keep
    for writer in ("tcgen05_sketch", "tcgen05_exact", "simt", "masked_ce"):
        keep = _write(writer, X, bank)
        val, idx = ops.score_topk(X, bank, K=8, out=_poisoned(B, 8))
        assert ops.last_rescan_count(DEV) == 0, writer
        ref_v, ref_i = reference_topk(X, bank, 8)
        assert torch.equal(val, ref_v) and torch.equal(idx, ref_i), writer
        del keep


# ---- 2. the TOR / POR level words ------------------------------------------------------------------------------------

def _hier(levels, D):
    from tests.test_gpu_hier_rows import _setup
    h, _, train_index, n_levels, args, table, bank_train = _setup(levels, 8, D, 1)
    return dict(h=h, train_index=train_index, n_levels=n_levels, args=args, table=table, bank_train=bank_train, D=D)


def _hier_batch(hs, kind, B, seed):
    """hot: each row the sum of one train row from every level (every level's maximum well above a random one);
    cold: anti-aligned with such a sum on even rows, random on odd rows.  Labels mixed, padding rows included."""
    from tests.test_gpu_hier_rows import _mixed_targets
    g = torch.Generator().manual_seed(seed)
    ends = [0] + hs["args"]["level_end"]
    bs = hs["args"]["bank_sorted"].float().cpu()
    pick = [torch.randint(ends[l], ends[l + 1], (B,), generator=g) for l in range(hs["n_levels"]) if ends[l + 1] > ends[l]]
    x = sum(bs[p] for p in pick) + 0.05 * torch.randn(B, hs["D"], generator=g)
    if kind == "cold":
        x = -x
        x[1::2] = torch.randn(x[1::2].shape, generator=g)
    x = ops.normalize_rows(x.to(DEV))
    return x, _mixed_targets(hs["h"], B, seed).to(DEV)


def _hier_expected(hs, x, targets):
    """Oracle counters (per label's sub-batch, in bin L; padding rows nowhere) and the oracle's logits."""
    from tests.test_gpu_hier_rows import _oracle_bin, _oracle_logits
    h, train_index = hs["h"], hs["train_index"]
    N = len(h)
    logits = _oracle_logits(x, hs["bank_train"], train_index, N)
    want = torch.zeros((ops.HGR_HIER_MAX_CHAIN + 1, 4), dtype=torch.int64)
    tc = targets.cpu()
    for lab in sorted({int(t) for t in tc.tolist() if 0 <= t < N}):
        rows = (tc == lab).nonzero().flatten()
        want[len(h.c2p[lab]) + 1] += _oracle_bin(logits[rows], train_index, h, lab)
    return want, logits


def _hier_check(hs, x, targets, counts, lvl, top1, what):
    from tests.test_gpu_hier_rows import _check_winners
    want, logits = _hier_expected(hs, x, targets)
    assert torch.equal(counts.cpu(), want), (what, counts.cpu()[counts.cpu().any(1)], want[want.any(1)])
    try:
        _check_winners(logits, hs["train_index"], hs["h"], lvl, top1)
    except AssertionError as e:
        raise AssertionError("%s: %s" % (what, e)) from None


_HIERS = {}


def _hiers():
    if not _HIERS:
        from tests.test_gpu_hier_rows import _LEVELS12
        _HIERS["cfg2"] = _hier(_LEVELS12, 1024)
        _HIERS["small"] = _hier((3, 9, 40, 160), 1024)
    return _HIERS


# (hierarchy, batch kind, B): the largest B first (a regrown workspace would start zeroed), then smaller and larger
# batches, B off the 128-row tile, and n_levels changing between calls (12 <-> 4 levels: the words change stride)
_HIER_SEQ = [("cfg2", "hot", 512), ("cfg2", "cold", 129), ("cfg2", "hot", 300), ("small", "cold", 300),
             ("small", "hot", 512), ("cfg2", "cold", 512), ("small", "cold", 5), ("cfg2", "cold", 257)]


def test_hier_rows_sequence_of_batches():
    hs_all = _hiers()
    for i, (name, kind, B) in enumerate(_HIER_SEQ):
        hs = hs_all[name]
        x, t = _hier_batch(hs, kind, B, seed=10 + i)
        counts = ops.new_hier_counts(DEV)
        lvl = torch.full((B, hs["n_levels"]), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
        top1 = torch.full((B,), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
        ops.hier_metrics_fused_rows(x, targets=t, counts=counts, lvl_idx=lvl, top1=top1, **hs["args"], **hs["table"])
        _hier_check(hs, x, t, counts, lvl, top1, "call %d (%s, %s, B = %d)" % (i, name, kind, B))


# (batch kind, B, where the two logical shards cut the sorted train bank: 1.0 = shard 1 empty, 0.0 = shard 0 empty)
_SHARD_SEQ = [("hot", 512, 1.0), ("cold", 300, 0.5), ("hot", 129, 0.0), ("cold", 512, 0.5), ("cold", 257, 1.0)]


@pytest.mark.parametrize("name", ["cfg2", "small"])
def test_hier_sharded_sequence_of_batches(name):
    """``hier_level_scatter`` by G = 2 logical shards on one stream, then ``hier_finish_rows_gathered`` over both
    shards' words; a shard without train rows in one call and with rows in the next, and the reverse."""
    from hgrnet_b200.dist import local_level_ends
    hs = _hiers()[name]
    a = hs["args"]
    M = a["bank_sorted"].shape[0]
    L = hs["n_levels"]
    for i, (kind, B, cut) in enumerate(_SHARD_SEQ):
        x, t = _hier_batch(hs, kind, B, seed=40 + i)
        parts = torch.full((2, B, L), -1, dtype=torch.int64, device=DEV)
        m = int(M * cut)
        for r, (lo, hi) in enumerate(((0, m), (m, M))):
            ops.hier_level_scatter(x, a["bank_sorted"][lo:hi], local_level_ends(a["level_end"], lo, hi), lo,
                                   [parts[r].data_ptr()], B)
        counts = ops.new_hier_counts(DEV)
        lvl = torch.full((B, L), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
        top1 = torch.full((B,), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
        ops.hier_finish_rows_gathered(parts.data_ptr(), 2, B * L, B, M, L, a["sorted_to_pos"], a["first_out"], t,
                                      hs["table"]["chain_ptr"], hs["table"]["chain_pos"], hs["table"]["chain_level"],
                                      counts, lvl_idx=lvl, top1=top1)
        _hier_check(hs, x, t, counts, lvl, top1, "call %d (%s, B = %d, cut %g)" % (i, kind, B, cut))


# ---- 3. the graph-replayed evaluators, a different batch every step -------------------------------------------------

def _check_lists(val, idx, x, bank, col_id, what):
    """Production lists of a graph step against the reference: a row that differs (re-scanned on the CUDA cores)
    must pass the float64 check."""
    ref_v, ref_i = reference_topk(x, bank, K, col_id=col_id)
    bad = (~((val == ref_v).all(1) & (idx == ref_i).all(1))).nonzero().flatten()
    try:
        check_topk_f64(val, idx, x, bank, K, col_id=col_id, rows=bad)
    except AssertionError as e:
        raise AssertionError("%s: %s" % (what, e)) from None


def test_eval_stream_hier_and_classes_new_batch_every_step(tmp_path):
    from hgrnet_b200.evaluate import HierMetrics
    from oracle import cases
    from tests.test_gpu_hier_rows import _model
    spec = cases.EVAL_CASES[1]
    model, h, _ = _model(spec, tmp_path)
    N, B, slots = len(h), spec["B"], 4
    es = model.make_eval_stream(batch=B, slots=slots, streams=3, hier_metrics=True, class_metrics=True)
    bank, col_id = model.bank_test, model._test_index_i32
    g = torch.Generator().manual_seed(8)
    batches = []
    for step in range(8):
        pick = torch.randint(0, bank.shape[0], (B,), generator=g)
        f = bank.float().cpu()[pick] + 0.02 * torch.randn(B, bank.shape[1], generator=g)
        if step % 2:
            f = -f
            f[1::2] = torch.randn(f[1::2].shape, generator=g)
        lab = col_id.cpu()[pick].int() if step % 2 == 0 else torch.randint(0, N, (B,), generator=g, dtype=torch.int32)
        lab[step % B] = -1
        batches.append((f, lab))
    es.begin()
    for step, (f, lab) in enumerate(batches):
        s = step % slots
        es.synchronize()
        es.host_feats[s].copy_(f)
        es.host_labels[s].copy_(lab)
        es.step(s)
        es.synchronize()
        _check_lists(es.val[s], es.idx[s], ops.normalize_rows(f.to(DEV)), bank, col_id, "step %d" % step)
    es.end()

    hits = ops.new_hits(DEV)
    hm = HierMetrics(model)
    classes = ops.new_class_counts(DEV, N)
    for f, lab in batches:
        x, t = ops.normalize_rows(f.to(DEV)), lab.to(DEV)
        _, idx = ops.score_topk(x, bank, col_id=col_id, targets=t, K=K, hits=hits)
        hm.update_rows(x, t)
        ops.class_hits(idx, t, classes)
    assert es.hit_counts() == hits.tolist()
    rows = 8 * (B - 1)
    assert hm.path_all_count == rows
    got, want = es.hier_ratios(), hm.ratios(rows)
    assert all(abs(a - b) < 1e-9 for a, b in zip(got, want)), (got, want)
    assert torch.equal(es.class_table().reshape(classes.shape), classes.cpu())


def _cfg2_bank():
    case = _case(*SHAPES[0])
    C = case["bank"].shape[0]
    col_id = torch.randperm(3 * C, generator=torch.Generator().manual_seed(4))[:C].int().to(DEV)
    return case["bank"], col_id


def _cfg2_batches(bank, col_id, n, seed):
    """Raw features of alternating hot / cold batches, with labels (ids of the bank rows they sit near on hot
    batches)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for i in range(n):
        x = (_hot if i % 2 == 0 else _cold)(bank, SHAPES[0][0], seed + i).float()
        f = 3.0 * x + 1e-3 * torch.randn(x.shape, generator=g).to(DEV)
        lab = col_id[(reference_topk(x.to(torch.bfloat16), bank, 1)[1][:, 0]).long()]
        lab[::5] = -1
        out.append((f, lab.int()))
    return out


def test_eval_stream_grid_share_new_batch_every_step():
    """``EvalStream`` at the grid share it picks for cfg 2 (2: two batches side by side on two streams)."""
    from hgrnet_b200.stream import EvalStream
    bank, col_id = _cfg2_bank()
    B = SHAPES[0][0]
    es = EvalStream(bank, col_id, batch=B, slots=4, streams=2, host_io=False)
    assert es.grid_share == 2
    batches = _cfg2_batches(bank, col_id, 8, seed=50)
    for step, (f, lab) in enumerate(batches):
        s = step % 4
        es.synchronize()
        es.dev_feats[s].copy_(f)
        es.dev_labels[s].copy_(lab)
        es.begin()
        es.step(s)
        es.synchronize()
        _check_lists(es.val[s], es.idx[s], ops.normalize_rows(f), bank, col_id, "step %d" % step)
    es.end()
    hits = ops.new_hits(DEV)
    for f, lab in batches:
        ops.score_topk(ops.normalize_rows(f), bank, col_id=col_id, targets=lab, K=K, hits=hits)
    assert es.hit_counts() == hits.tolist()


def test_sharded_eval_stream_one_rank_new_batches_every_run():
    from hgrnet_b200.dist import ShardedEvalStream
    bank, col_id = _cfg2_bank()
    B = SHAPES[0][0]
    ses = ShardedEvalStream(bank, 0, batch=B, K=K, steps=8, col_id=col_id, host_io=False)
    hits = ops.new_hits(DEV)
    try:
        for run in range(2):
            batches = _cfg2_batches(bank, col_id, 8, seed=70 + 10 * run)
            if run:
                batches = batches[1:] + batches[:1]          # each slot changes kind between the two runs
            torch.cuda.synchronize()
            for s, (f, lab) in enumerate(batches):
                ses.dev_feats[s].copy_(f)
                ses.dev_labels[s].copy_(lab)
            ses.run()
            torch.cuda.synchronize()
            for s, (f, lab) in enumerate(batches):
                _check_lists(ses.val[s], ses.idx[s], ops.normalize_rows(f), bank, col_id, "run %d step %d" % (run, s))
                ops.score_topk(ops.normalize_rows(f), bank, col_id=col_id, targets=lab, K=K, hits=hits)
        assert ses.all_reduce_hits().tolist() == hits.tolist()
    finally:
        ses.close()


# ---- 4. the host-side plan cache of the grouped schedule -------------------------------------------------------------

def _split_refs(X, bank, ends, masks, S):
    starts = [0] + list(ends[:-1])
    out = []
    for s in range(S):
        rows = torch.cat([torch.arange(a, e) for a, e, m in zip(starts, ends, masks) if (m >> s) & 1]).to(DEV)
        out.append((rows, reference_topk(X, bank[rows].contiguous(), K, col_id=rows.int())))
    return out


def test_plan_cache_split_totals_of_the_class_shard():
    """Only ``split_C_total`` differs between calls: the list length follows it, and with G = 1 the certified merge
    gives every split's reference (re-scanned rows: float64)."""
    B, C, D = 512, 4000, 256
    X, bank = _rand(B, D, 90), _rand(C, D, 91)
    ends, masks = [1200, 2800, 4000], [1, 3, 2]
    cs = [2800, 2800]
    totals = [cs, [2 * cs[0], 2 * cs[1]], [8 * cs[0], 8 * cs[1]], [cs[0], 8 * cs[1]], cs]
    kls = [ops.splits_global_list_len(B, C, D, K, ends, masks, tot) for tot in totals]
    assert len(set(kls)) >= 2 and kls[0] == kls[-1], kls
    refs = _split_refs(X, bank, ends, masks, 2)
    table = ops.shard_table([(bank.data_ptr(), 0, C, 0)], DEV)
    node_splits = torch.ones(C, dtype=torch.uint8, device=DEV)
    stride = 2 * B * K + B                       # a split's area: its lists and bounds (the ABI's minimum)
    for tot in totals:
        v = torch.full((2 * stride,), float("nan"), device=DEV)
        i = torch.full((2 * stride,), 0x7FFFFFFF, dtype=torch.int32, device=DEV)
        bnd = torch.full((2 * stride,), float("nan"), device=DEV)
        ops.score_topk_splits_scatter(X, bank, ends, masks, tot, [v.data_ptr()], [i.data_ptr()], [bnd.data_ptr()], B,
                                      stride)
        repairs = torch.zeros(1, dtype=torch.int32, device=DEV)
        val, idx = ops.topk_merge_splits_certified(v.data_ptr(), i.data_ptr(), bnd.data_ptr(), 1, B, K, 2, B * K, B,
                                                   stride, X, table, node_splits, DEV, repair_count=repairs)
        for s, (rows, (ref_v, ref_i)) in enumerate(refs):
            bad = (~((val[s] == ref_v).all(1) & (idx[s] == ref_i).all(1))).nonzero().flatten()
            assert bad.numel() <= int(repairs.item()), (tot, s, bad.numel(), int(repairs.item()))
            check_topk_f64(val[s], idx[s], X, bank[rows].contiguous(), K, col_id=rows.int(), rows=bad)


def test_plan_cache_more_group_tables_than_slots():
    """Ten group tables over the same (B, C, D, K) -- more than the cache's 8 slots -- then the first again, and the
    same ends with other split bits: every call equals the reference of each of its splits."""
    B, C, D = 64, 1000, 64
    X, bank = _rand(B, D, 92), _rand(C, D, 93)
    tables = [([100 * (j + 1), 500 + 30 * j, C], [1, 3, 2]) for j in range(4)]
    tables += [([17 + j, C], [3, 1]) for j in range(3)]
    tables += [([250, 500, 750, C], [1, 2, 1, 3]), ([C // 2, C], [1, 2]), ([1, 2, 3, C], [3, 2, 1, 3])]
    tables += [tables[0], (tables[0][0], [2, 1, 3]), (tables[0][0], [3, 3, 1])]
    for impl in ("tcgen05_exact", "tcgen05"):
        for n, (ends, masks) in enumerate(tables):
            val, idx = ops.score_topk_splits(X, bank, ends, masks, 2, K=K, impl=_impl(impl), out=_poisoned(B, K, 2))
            rescans = ops.last_rescan_count(DEV) if impl == "tcgen05" else 0
            for s, (rows, (ref_v, ref_i)) in enumerate(_split_refs(X, bank, ends, masks, 2)):
                bad = (~((val[s] == ref_v).all(1) & (idx[s] == ref_i).all(1))).nonzero().flatten()
                assert bad.numel() <= rescans, (impl, n, ends, masks, s, bad.numel(), rescans)
                check_topk_f64(val[s], idx[s], X, bank[rows].contiguous(), K, col_id=rows.int(), rows=bad)
