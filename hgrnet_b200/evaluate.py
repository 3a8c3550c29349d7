"""Re-hosted eval loop of the reference (``main.test``, main.py:104-222).

Per batch the reference materialises logits [B,N], gathers the test columns, runs
``topk(20)``, maps ids, compares with the label and sums Hit@{1,2,5,10,20} (main.py:135-147).
Here that whole chain is ONE fused call, ``model.score_topk`` (kernel (1) + kernel (2)); the
hit counters stay on the device until the loop ends, as in the reference.  The hierarchical
metrics TOR / POR (``hit_ratio`` / ``path_ratio`` / ``point_ratio``, main.py:143,152-191) are the
first "next" row of SURVEY.md section 8f: a per-level arg-max in the epilogue of the GEMM against
the level-sorted train bank, then chain matching on the device (``hgr_hier_metrics_fused_rows``);
no per-sample python loop, no D2H copies.
Output format: ``count_acc`` (utils.py:135-146) and the log files of main.py:205-222.
"""
from __future__ import annotations

import copy
import itertools
from typing import Iterable, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops
from ._cabi import HGR_HIER_MAX_CHAIN, HGR_MISTAKE_COUNTERS, HIT_CUTS


def count_acc(hits_dict, num_tot):
    """utils.py:135-146."""
    out_str = ""
    acc_dict = dict()
    keys = list(hits_dict.keys())
    for key, value in hits_dict.items():
        acc = value / num_tot * 100.0
        acc_dict[key] = acc
        out_str += "Top@{}(%):{:.2f}".format(key, acc)
        out_str += ", " if key != keys[-1] else "."
    return out_str, acc_dict


def chain_csr(c2p: Sequence[Sequence[int]]) -> Tuple[np.ndarray, np.ndarray]:
    """A CSR over all nodes whose row n is the reference's label chain ``c2p[n] + [n]`` (main.py:152): int64
    ``(chain_ptr [N + 1], nodes)``, the node ids of every chain.  ``hgr_hier_mistakes`` takes it as it is (as int32)."""
    n = len(c2p)
    lens = np.fromiter((len(c) + 1 for c in c2p), dtype=np.int64, count=n)
    chain_ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=chain_ptr[1:])
    nodes = np.fromiter(itertools.chain.from_iterable((*c, i) for i, c in enumerate(c2p)), dtype=np.int64,
                        count=int(chain_ptr[-1]))
    return chain_ptr, nodes


def chain_table(c2p: Sequence[Sequence[int]], depth: np.ndarray, train_ids: Sequence[int]
                ) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """The chain table of ``hgr_hier_metrics_fused_rows``: the CSR of ``chain_csr``.  Returns int32 ``(chain_ptr
    [N + 1], chain_pos, chain_level)``: per entry the node's position in ``train_ids`` (the last one if it repeats, -1 if
    it is not a train class) and its depth."""
    n = len(c2p)
    chain_ptr, nodes = chain_csr(c2p)
    pos_of = np.full(n, -1, dtype=np.int64)
    train = np.asarray(train_ids, dtype=np.int64)
    pos_of[train] = np.arange(train.size)                # repeated ids: the last assignment stays, as in a dict
    return (chain_ptr.astype(np.int32), pos_of[nodes].astype(np.int32),
            np.asarray(depth, dtype=np.int64)[nodes].astype(np.int32))


_TOTALS_DIV = {}


def hier_totals(counts: torch.Tensor) -> torch.Tensor:
    """Per-chain-length counters (``ops.new_hier_counts``: bin L = {rows, TOR hits, points, edges}) -> float64 ``[4]``
    ``(rows, hits, point, path)`` on the counters' device: the sums the reference adds to ``path_all_count``,
    ``hits_all``, ``point_all`` and ``path_all`` (main.py:158-191), with ``point = sum_L points_L / L`` and
    ``path = sum_L edges_L / max(L - 1, 1)``.  ``[S, L, 4]`` counters give ``[S, 4]``.  No host synchronisation."""
    div = _TOTALS_DIV.get(counts.device)
    if div is None or div.shape[0] != counts.shape[-2]:
        L = torch.arange(counts.shape[-2], dtype=torch.float64)
        one = torch.ones_like(L)
        div = torch.stack([one, one, L.clamp(min=1), (L - 1).clamp(min=1)], 1).to(counts.device)
        _TOTALS_DIV[counts.device] = div
    return (counts.double() / div).sum(-2)


def hier_line(hit_ratio: float, path_ratio: float, point_ratio: float) -> str:
    """The TOR / POR suffix of the reference's ``test()`` line (main.py:205-214), ratios in percent."""
    return " hit_ratio(%):{:.2f} path_ratio(%):{:.2f} point_ratio(%):{:.2f}".format(hit_ratio, path_ratio, point_ratio)


class HierMetrics:
    """TOR / POR counters (main.py:123-127,152-191).  One fused call per batch (``hgr_hier_metrics_fused_rows``):
    per-level arg-max over the train classes in the epilogue of the GEMM against the level-sorted train bank, then
    chain matching and counting on the device into integer counters per chain length (``counts``), incremented in
    place; nothing is copied to the host before the ratios are printed.

    ``update_rows`` scores every row against its own label and needs no host work per batch."""

    def __init__(self, model):
        self.model = model
        dev = model.device
        self.counts = ops.new_hier_counts(dev)
        depth = torch.from_numpy(model.hierarchy.depth).to(torch.int64)
        self.n_levels = int(depth.max()) + 1 if depth.numel() else 1
        # Only the TRAIN columns enter TOR / POR (main.py:143,155,174): the GEMM runs against the train rows of the bank
        # alone (M = 983 of 18,278 classes on ImageNet-21K-D) instead of all N nodes, and the kernels work in train
        # POSITIONS: the label's chain as positions (-1: not a train class).
        train = model.train_index.cpu()
        dt = depth[train]
        M = dt.numel()
        # first position of train_index that is NOT at level l: where the reference's -1 fill (main.py:171) sits first
        first_out = []
        for l in range(self.n_levels):
            out = (dt != l).nonzero()
            first_out.append(int(out[0]) if out.numel() else M)
        self._first_out = torch.tensor(first_out, dtype=torch.int32, device=dev)
        # the train rows of the bank sorted by level -- stable, so that inside a level the sorted order is the
        # train_index order and "first position among equal values" is preserved
        order = torch.sort(dt, stable=True).indices
        self._sorted_to_pos = order.to(torch.int32).to(dev)
        self._level_end = torch.cumsum(torch.bincount(dt, minlength=self.n_levels), 0).tolist()
        self._bank_sorted = None      # built on first use from model.bank_train (update_classifier must have run)
        self._bank_version = None
        self._train_ids = train.tolist()
        self._chains = None           # chain table of update_rows, built on first use

    @property
    def path_all_count(self) -> int:
        """Rows scored so far (synchronises)."""
        return int(self.counts[:, 0].sum())

    def sorted_bank(self) -> torch.Tensor:
        """The train rows of the bank sorted by level; re-sorted when ``model.bank_train`` was refreshed (new tensor or
        in-place update)."""
        bank = self.model.bank_train
        stamp = (bank.data_ptr(), bank._version)
        if self._bank_sorted is None or self._bank_version != stamp:
            self._bank_sorted = bank[self._sorted_to_pos.long()].contiguous()
            self._bank_version = stamp
        return self._bank_sorted

    def rows_args(self) -> dict:
        """Every argument of ``ops.hier_metrics_fused_rows`` except the batch (``x_norm``, ``targets``) and the
        counters.  Device tensors; the chain table is built on the first call."""
        if self._chains is None:
            m = self.model
            dev = self._first_out.device
            self._chains = tuple(torch.from_numpy(a).to(dev)
                                 for a in chain_table(m.c2p, m.hierarchy.depth, self._train_ids))
        chain_ptr, chain_pos, chain_level = self._chains
        return dict(bank_sorted=self.sorted_bank(), level_end=self._level_end, sorted_to_pos=self._sorted_to_pos,
                    first_out=self._first_out, chain_ptr=chain_ptr, chain_pos=chain_pos, chain_level=chain_level)

    def update_rows(self, x_norm: torch.Tensor, targets: torch.Tensor, node_splits: Optional[torch.Tensor] = None,
                    counts: Optional[torch.Tensor] = None):
        """Score a batch: ``x_norm`` [B, D] bf16 normalised image features, row i scored against the chain of node
        ``targets[i]``, so a batch may mix classes.  Rows whose target lies outside ``[0, n_nodes)`` are skipped
        (padding).  Into ``counts`` (default: the object's own); with ``node_splits``, ``counts`` ``[S, 33, 4]`` takes
        one set per split (``ops.hier_metrics_fused_rows``).  No host work per batch and no synchronisation."""
        ops.hier_metrics_fused_rows(x_norm, targets=targets.to(torch.int32), node_splits=node_splits,
                                    counts=self.counts if counts is None else counts, **self.rows_args())

    def ratios(self, num_sample):
        """``(hit_ratio, path_ratio, point_ratio)`` of the reference's line: TOR and POR over all ``num_sample`` rows,
        the path ratio over the rows in the hierarchy (synchronises)."""
        rows, hits, point, path = hier_totals(self.counts).tolist()
        return hits / num_sample * 100.0, path / rows * 100.0, point / num_sample * 100.0


def mistake_summary(counts, K: int = 20) -> dict:
    """The derived values of one set of ``hier_mistakes`` counters (``[HGR_MISTAKE_COUNTERS]``, tensor or list), as
    float64: ``rows``, ``mistakes``, ``mistake_rate`` = mistakes / rows, ``severity_h`` / ``severity_d`` = the sum of
    h / d at top-1 over the mistakes (0 without mistakes; a correct top-1 adds 0), ``hdist@k`` / ``dist@k`` = the sum of
    h / d over the first min(k, K) entries / (rows * min(k, K)), and ``hist_d`` the histogram of d at top-1 (last bin:
    larger than 2 * HGR_HIER_MAX_CHAIN).  ``K`` is the list length.  All zero without rows."""
    c = [int(v) for v in (counts.tolist() if hasattr(counts, "tolist") else counts)]
    if len(c) != HGR_MISTAKE_COUNTERS:
        raise ValueError("one set of %d mistake counters expected, got %d" % (HGR_MISTAKE_COUNTERS, len(c)))
    rows, mistakes = float(c[0]), float(c[1])
    nh = len(HIT_CUTS)
    out = {"rows": rows, "mistakes": mistakes, "mistake_rate": mistakes / rows if rows else 0.0,
           "severity_h": c[2] / mistakes if mistakes else 0.0, "severity_d": c[2 + nh] / mistakes if mistakes else 0.0}
    for i, k in enumerate(HIT_CUTS):
        n = rows * min(k, K)
        out["hdist@%d" % k] = c[2 + i] / n if n else 0.0
        out["dist@%d" % k] = c[2 + nh + i] / n if n else 0.0
    out["hist_d"] = [float(v) for v in c[2 + 2 * nh:]]
    return out


def mistake_line(summary: dict) -> str:
    """The suffix ``test()`` appends to its line with ``--hgr_mistake_metrics``."""
    return " mistake_rate(%):{:.2f} severity:{:.2f} hdist@1:{:.2f} hdist@5:{:.2f} hdist@20:{:.2f}".format(
        summary["mistake_rate"] * 100.0, summary["severity_h"], summary["hdist@1"], summary["hdist@5"],
        summary["hdist@20"])


class MistakeMetrics:
    """Hierarchical mistake severity and LCA distance@k (Bertinetto et al., "Making Better Mistakes", CVPR 2020) of
    the top-K lists of every batch: how far from the label in the hierarchy the predictions are, not only whether the
    label is among them (main.py:135-148).  Holds the chain table (``chain_csr`` of ``model.c2p``, on the device) and
    the counters, one set per list set; ``update`` counts a batch on the device (``ops.hier_mistakes``) with no host
    synchronisation.  ``n_sets`` > 1 counts ``[n_sets, B, K]`` lists of several test splits (``SplitEval``).
    ``counts``: the ``[n_sets, HGR_MISTAKE_COUNTERS]`` counters to own (default: new ones), e.g. a view of an
    ``EvalCounters`` block."""

    def __init__(self, model, n_sets: int = 1, K: int = 20, counts: Optional[torch.Tensor] = None):
        dev = model.device
        ptr, nodes = chain_csr(model.c2p)
        self.chain_ptr = torch.from_numpy(ptr.astype(np.int32)).to(dev)
        self.chain_node = torch.from_numpy(nodes.astype(np.int32)).to(dev)
        self.n_sets, self.K = n_sets, K
        self.counts = ops.new_mistake_counts(dev, n_sets) if counts is None else counts

    def args(self) -> dict:
        """The chain table arguments of ``ops.hier_mistakes``."""
        return dict(chain_ptr=self.chain_ptr, chain_node=self.chain_node)

    def update(self, idx: torch.Tensor, targets: torch.Tensor, node_splits: Optional[torch.Tensor] = None,
               counts: Optional[torch.Tensor] = None):
        """Count a batch: ``idx`` int32 node ids ``[B, K]`` (or ``[n_sets, B, K]`` with ``node_splits``), ``targets``
        [B] node ids, one per row (-1 padding counts nowhere).  Into ``counts`` (default: the object's own)."""
        ops.hier_mistakes(idx, targets.to(torch.int32), counts=self.counts if counts is None else counts,
                          node_splits=node_splits, **self.args())

    def summary(self, counts: Optional[torch.Tensor] = None):
        """``mistake_summary`` of every set (synchronises): a dict, or a list of dicts for several sets."""
        c = (self.counts if counts is None else counts).view(-1, HGR_MISTAKE_COUNTERS).tolist()
        out = [mistake_summary(x, self.K) for x in c]
        return out[0] if self.n_sets == 1 else out


def class_summary(table) -> dict:
    """The class-averaged Hit@k of one set's per-class table (``[n_nodes, HGR_NUM_HITS + 1]`` int64 rows
    ``[Hit@1, Hit@2, Hit@5, Hit@10, Hit@20, rows]``, tensor or array), as floats: ``classes`` = the number of classes
    with at least one row, and ``mean@k`` for k in ``HIT_CUTS`` = the mean over those classes of Hit@k / rows (every
    class weighs the same, whatever its row count).  All zero without rows."""
    t = np.asarray(table.cpu() if hasattr(table, "cpu") else table, dtype=np.int64)
    if t.ndim != 2 or t.shape[1] != len(HIT_CUTS) + 1:
        raise ValueError("one set of per-class counters [n_nodes, %d] expected, got %s" % (len(HIT_CUTS) + 1,
                                                                                           list(t.shape)))
    rows = t[:, -1]
    seen = rows > 0
    n = int(seen.sum())
    mean = (t[seen, :-1] / rows[seen, None]).mean(0) if n else np.zeros(len(HIT_CUTS))
    out = {"classes": float(n)}
    for k, m in zip(HIT_CUTS, mean.tolist()):
        out["mean@%d" % k] = float(m)
    return out


def class_line(summary: dict) -> str:
    """The suffix ``test()`` appends to its line with ``--hgr_class_metrics``, in percent:
    ``" class_mean Top@1(%):xx.xx, Top@2(%):xx.xx, Top@5(%):xx.xx, Top@10(%):xx.xx, Top@20(%):xx.xx over N classes"``."""
    return " class_mean " + ", ".join("Top@{}(%):{:.2f}".format(k, summary["mean@%d" % k] * 100.0) for k in HIT_CUTS) \
        + " over {} classes".format(int(summary["classes"]))


class ClassHits:
    """Per-class Hit@{1,2,5,10,20} and row counts of the top-K lists of every batch, the table behind the
    class-averaged Hit@k (``class_summary``) that zero-shot results on ImageNet are usually compared by (e.g. Xian et
    al., TPAMI 2018): the reference's test loader holds one class per batch, so its image-weighted Hit@k
    (main.py:135-148) is dominated by the most populous classes.  Holds the counters ``[n_sets, n_nodes,
    HGR_NUM_HITS + 1]``; ``update`` counts a batch on the device (``ops.class_hits``) with no host synchronisation.
    ``n_sets`` > 1 counts ``[n_sets, B, K]`` lists of several test splits (``SplitEval``).  ``counts``: the counters to
    own (default: new ones)."""

    def __init__(self, model, n_sets: int = 1, K: int = 20, counts: Optional[torch.Tensor] = None):
        self.n_nodes = len(model.nodes)
        self.n_sets, self.K = n_sets, K
        self.counts = ops.new_class_counts(model.device, self.n_nodes, n_sets) if counts is None else counts

    def update(self, idx: torch.Tensor, targets: torch.Tensor, node_splits: Optional[torch.Tensor] = None,
               counts: Optional[torch.Tensor] = None):
        """Count a batch: ``idx`` int32 node ids ``[B, K]`` (or ``[n_sets, B, K]`` with ``node_splits``), ``targets``
        [B] node ids, one per row (-1 padding counts nowhere).  Into ``counts`` (default: the object's own)."""
        ops.class_hits(idx, targets.to(torch.int32), self.counts if counts is None else counts, node_splits=node_splits)

    def table(self) -> torch.Tensor:
        """The host int64 table so far (synchronises): ``[n_nodes, 6]``, or ``[n_sets, n_nodes, 6]`` for several sets."""
        t = self.counts.cpu()
        return t[0] if self.n_sets == 1 else t

    def summary(self):
        """``class_summary`` of every set (synchronises): a dict, or a list of dicts for several sets."""
        out = [class_summary(t) for t in self.counts.cpu()]
        return out[0] if self.n_sets == 1 else out


_BANK_SEED = 0x48475221   # the seed of tree_model's test-bank permutation (head.py)


def split_groups(splits, n_nodes: int):
    """Host layout of the multi-split bank.  ``splits``: ``{name: node ids}`` (at most 8).  Every class of the union
    gets the bit mask of the splits that hold it; classes of equal mask form one GROUP, groups in ascending mask order,
    and inside a group the rows follow a fixed pseudo-random permutation (as ``tree_model``'s test bank does, so that an
    image's top-20 are not packed into a few adjacent rows).  Returns ``(names, bank_nodes int64 [C], group_end,
    group_splits, node_splits uint8 [n_nodes])``."""
    names = list(splits)
    if not 1 <= len(names) <= 8:
        raise ValueError("between 1 and 8 splits, got %d" % len(names))
    node_splits = np.zeros(n_nodes, dtype=np.uint8)
    for s, name in enumerate(names):
        ids = np.asarray(list(splits[name]), dtype=np.int64)
        if ids.size == 0:
            raise ValueError("split %r is empty" % name)
        node_splits[ids] |= np.uint8(1 << s)
    masks = sorted(set(node_splits[node_splits != 0].tolist()))
    if len(masks) > 16:
        raise ValueError("%d groups of equal split membership; at most 16" % len(masks))
    gen = torch.Generator().manual_seed(_BANK_SEED)
    rows, group_end = [], []
    for m in masks:
        ids = np.nonzero(node_splits == m)[0]
        perm = torch.randperm(ids.size, generator=gen).numpy() if ids.size > 1 else np.zeros(1, dtype=np.int64)
        rows.append(ids[perm])
        group_end.append((group_end[-1] if group_end else 0) + ids.size)
    return names, np.concatenate(rows), group_end, masks, node_splits


def split_line(name, hits, rows, hier=None, mistakes=None, classes=None):
    """The reference's ``test()`` line of one split (``count_acc`` + TOR / POR), prefixed with the split's name.
    ``hier``: ``(hits, point, path, path_rows)`` sums or None; ``mistakes``: the split's ``mistake_summary`` or None;
    ``classes``: the split's ``class_summary`` or None."""
    out_str, _ = count_acc(dict(zip(HIT_CUTS, hits)), rows)
    if hier is not None:
        tor, point, path, path_rows = hier
        out_str += hier_line(tor / rows * 100.0, path / path_rows * 100.0 if path_rows else 0.0, point / rows * 100.0)
    if mistakes is not None:
        out_str += mistake_line(mistakes)
    if classes is not None:
        out_str += class_line(classes)
    return "{}: {}".format(name, out_str)


class EvalCounters:
    """The integer counters of one evaluator in ONE int64 device buffer (``counters``), and every value reported from
    them.  Layout: ``hits [HGR_NUM_HITS]`` (Hit@{1,2,5,10,20}); with S splits ``split_counts [S, HGR_NUM_HITS + 1]``
    (per split Hit@k and rows); with ``hier`` ``hier_counts [n, HGR_HIER_MAX_CHAIN + 1, 4]`` (TOR / POR per chain
    length); with ``mistakes`` ``mistake_counts [n, HGR_MISTAKE_COUNTERS]`` -- n = S, or 1 without splits.  The
    kernels increment the views in place, so nothing is zeroed per batch and a stream mirrors everything to the host
    with one copy.  ``read(counters)`` gives the counters the readout reports, in the same layout (default: the
    buffer itself): a stream synchronises its streams first, a class-sharded stream also sums them over ranks.

    With ``classes`` (the node count) the per-class table ``class_counts [n, classes, HGR_NUM_HITS + 1]``
    (``ClassHits``) is a buffer of its own, outside ``counters``: at 21,841 nodes it is 1 MB per set, and the streams
    copy ``counters`` to the host after every step.  It is read only by the readout, through the same ``read``."""

    def __init__(self, device, n_splits: int = 0, hier: bool = False, mistakes: bool = False, K: int = 20, read=None,
                 classes: int = 0):
        n = max(n_splits, 1)
        self.S, self.K = n_splits, K
        self._shapes = [(ops.HGR_NUM_HITS,), (n_splits, ops.HGR_NUM_HITS + 1),
                        (n if hier else 0, HGR_HIER_MAX_CHAIN + 1, 4), (n if mistakes else 0, HGR_MISTAKE_COUNTERS)]
        self.counters = torch.zeros(sum(int(np.prod(sh)) for sh in self._shapes), dtype=torch.int64, device=device)
        self.hits, self.split_counts, self.hier_counts, self.mistake_counts = self._views(self.counters)
        self.class_counts = ops.new_class_counts(device, classes, n) if classes else None
        self._read = read

    def zero_(self):
        """Zero every counter (a stream does so after its warm-up runs)."""
        self.counters.zero_()
        if self.class_counts is not None:
            self.class_counts.zero_()

    def _views(self, counters: torch.Tensor):
        parts = torch.split(counters, [int(np.prod(sh)) for sh in self._shapes])
        return tuple(p.view(sh) if p.numel() else None for p, sh in zip(parts, self._shapes))

    def read(self):
        """``(hits, split_counts, hier_counts, mistake_counts)`` to report, after the read step."""
        return self._views(self.counters if self._read is None else self._read(self.counters))

    def _need(self, what: str, have: bool):
        if not have:
            raise RuntimeError("the evaluator was built without %s" % what)

    def hit_counts(self):
        """Hit@{1,2,5,10,20} so far."""
        return self.read()[0].tolist()

    def split_hit_counts(self):
        """Per split ``[Hit@1, @2, @5, @10, @20, rows]`` so far, in split order."""
        self._need("splits", self.S > 0)
        return self.read()[1].tolist()

    def split_ratios(self):
        """Per counter set ``(hit_ratio, path_ratio, point_ratio)`` in percent -- the TOR / POR of the reference's
        ``test()`` line -- over the rows of the set whose label lies in the hierarchy (0 without rows)."""
        self._need("TOR / POR counters", self.hier_counts is not None)
        return [(0.0, 0.0, 0.0) if rows == 0 else (hits / rows * 100.0, path / rows * 100.0, point / rows * 100.0)
                for rows, hits, point, path in hier_totals(self.read()[2]).tolist()]

    def hier_ratios(self):
        """``split_ratios`` of the one set without splits."""
        self._need("TOR / POR counters without splits", self.S == 0)
        return self.split_ratios()[0]

    def mistake_summary(self):
        """``mistake_summary`` of the one set without splits."""
        self._need("mistake counters without splits", self.mistake_counts is not None and self.S == 0)
        return mistake_summary(self.read()[3][0], self.K)

    def split_mistake_summary(self):
        """Per split ``mistake_summary`` over the rows whose label is in the split."""
        self._need("per-split mistake counters", self.mistake_counts is not None and self.S > 0)
        return [mistake_summary(c, self.K) for c in self.read()[3]]

    def class_table(self) -> torch.Tensor:
        """The per-class table so far as a host int64 tensor: ``[n_nodes, HGR_NUM_HITS + 1]`` without splits,
        ``[S, n_nodes, HGR_NUM_HITS + 1]`` with them (``hgr_class_hits``'s layout)."""
        self._need("per-class counters", self.class_counts is not None)
        t = (self.class_counts if self._read is None else self._read(self.class_counts)).cpu()
        return t if self.S > 0 else t[0]

    def class_summary(self):
        """``class_summary`` of the one set without splits."""
        self._need("per-class counters without splits", self.class_counts is not None and self.S == 0)
        return class_summary(self.class_table())

    def split_class_summary(self):
        """Per split ``class_summary`` over the rows whose label is in the split."""
        self._need("per-split per-class counters", self.class_counts is not None and self.S > 0)
        return [class_summary(t) for t in self.class_table()]

    def split_lines(self, names):
        """One ``split_line`` per split: Hit@k, plus TOR / POR, the mistake metrics and the class-averaged Hit@k when
        counted."""
        self._need("splits", self.S > 0)
        _, counts, hier, mist = self.read()
        hier = [None] * self.S if hier is None else [(tor, point, path, rows)
                                                     for rows, tor, point, path in hier_totals(hier).tolist()]
        mist = [None] * self.S if mist is None else [mistake_summary(c, self.K) for c in mist.tolist()]
        cls = [None] * self.S if self.class_counts is None else self.split_class_summary()
        return [split_line(name, c[:ops.HGR_NUM_HITS], max(c[ops.HGR_NUM_HITS], 1), h, m, k)
                for name, c, h, m, k in zip(names, counts.tolist(), hier, mist, cls)]


class SplitEval:
    """Several test splits of one hierarchy scored in ONE pass per batch (``hgr_score_topk_splits``): the union bank is
    built from ``model.zsl_weights`` in the group layout of ``split_groups`` and rebuilt after a bank refresh; the
    counters of every split stay on the device (``EvalCounters``: ``split_counts``, ``hier_counts``,
    ``mistake_counts``).  With ``hier=True`` the TOR / POR counters of every split follow from one level GEMM per batch
    (``HierMetrics.update_rows`` with ``node_splits``).  With ``mistakes=True`` the mistake severity and LCA
    distance@k of every split are counted from the ``[S, B, K]`` lists (``MistakeMetrics``, one set per split).  With
    ``class_metrics=True`` so is the per-class Hit@k table (``ClassHits``, one set per split; ``class_counts``).
    ``lines()`` gives one line per split."""

    def __init__(self, model, splits, hier: bool = True, K: int = 20, mistakes: bool = False,
                 class_metrics: bool = False):
        self.model = model
        self.K = K
        dev = model.device
        names, bank_nodes, self.group_end, self.group_splits, node_splits = split_groups(splits, len(model.nodes))
        self.names = names
        self.S = len(names)
        self._bank_nodes = torch.from_numpy(bank_nodes).to(dev)
        self.col_id = self._bank_nodes.to(torch.int32)
        self.node_splits = torch.from_numpy(node_splits).to(dev)
        self.tally = EvalCounters(dev, n_splits=self.S, hier=hier, mistakes=mistakes, K=K,
                                  classes=len(model.nodes) if class_metrics else 0)
        self.split_counts, self.hier_counts = self.tally.split_counts, self.tally.hier_counts
        self.mistake_counts = self.tally.mistake_counts
        self.hier = HierMetrics(model) if hier else None
        self.mistakes = MistakeMetrics(model, n_sets=self.S, K=K, counts=self.mistake_counts) if mistakes else None
        self.class_counts = self.tally.class_counts
        self.classes = ClassHits(model, n_sets=self.S, K=K, counts=self.class_counts) if class_metrics else None
        self._bank = None
        self._bank_version = None

    def bank(self) -> torch.Tensor:
        """The union bank in group layout; rebuilt when ``model.zsl_weights`` was refreshed (new tensor or in place)."""
        w = self.model.zsl_weights
        stamp = (w.data_ptr(), w._version)
        if self._bank is None or self._bank_version != stamp:
            self._bank = w.index_select(0, self._bank_nodes).contiguous()
            self._bank_version = stamp
        return self._bank

    def score_args(self) -> dict:
        return dict(bank=self.bank(), group_end=self.group_end, group_splits=self.group_splits, n_splits=self.S,
                    col_id=self.col_id, node_splits=self.node_splits, K=self.K)

    def update(self, x_norm: torch.Tensor, targets: torch.Tensor, hier_targets: Optional[torch.Tensor] = None):
        """Score a batch against every split: ``x_norm`` [B, D] bf16, ``targets`` [B] node ids (a row counts toward
        the splits its label belongs to).  TOR / POR match row i against ``hier_targets[i]`` (default: ``targets``).
        Returns ``(val [S,B,K], idx [S,B,K])``.  No host synchronisation."""
        t = targets.to(torch.int32)
        out = ops.score_topk_splits(x_norm, targets=t, counts=self.split_counts, **self.score_args())
        if self.hier is not None:
            self.hier.update_rows(x_norm, t if hier_targets is None else hier_targets, node_splits=self.node_splits,
                                  counts=self.hier_counts)
        if self.mistakes is not None:
            self.mistakes.update(out[1], t, node_splits=self.node_splits)
        if self.classes is not None:
            self.classes.update(out[1], t, node_splits=self.node_splits)
        return out

    def hit_counts(self):
        """Per split ``[Hit@1, @2, @5, @10, @20, rows]`` so far (synchronises)."""
        return self.tally.split_hit_counts()

    def lines(self):
        """One line per split: ``name: Top@1(%):..., ... .`` plus TOR / POR with ``hier``, the mistake metrics with
        ``mistakes`` and the class-averaged Hit@k with ``class_metrics`` (synchronises)."""
        return self.tally.split_lines(self.names)


def test(opts, model, device, splits=None, loader: Optional[Iterable] = None, log: bool = True):
    """Drop-in for main.py:104-222.  ``loader`` yields the reference's batch dicts
    ``{'img': [1,B,...], 'label': [1,B]}`` (single-label batches, imagenet_group_test.py).

    TOR / POR score every row of a batch against the batch's first label, as the reference does with ``targets[0]``
    (main.py:152).  A first label outside the hierarchy is counted nowhere (the reference raises ``IndexError``).
    With ``--hgr_mistake_metrics`` the line also gets the mistake rate, the mistake severity and the LCA distance@k
    (``MistakeMetrics``), every row against its own label.  With ``--hgr_class_metrics`` it also gets the
    class-averaged Hit@k (``ClassHits``, ``class_line``), every row counted toward its own label."""
    print("out", opts.out_ratio)
    print("in", opts.in_ratio)
    model.eval()
    model.update_classifier()
    if loader is None:
        raise ValueError("hgrnet_b200.evaluate.test needs a loader: image I/O (dataset/imagenet_group_test.py) is "
                         "an upstream component; pass loader=DataManager_test(...).get_data_loader()")
    print("Running.", flush=True)
    split_keys = [k for k in (getattr(opts, "hgr_eval_splits", "") or "").split(",") if k]
    if split_keys:
        return _test_splits(opts, model, device, splits, split_keys, loader, log)
    hier = HierMetrics(model) if getattr(opts, "hgr_hier_metrics", True) else None
    mist = MistakeMetrics(model) if getattr(opts, "hgr_mistake_metrics", False) else None
    cls = ClassHits(model) if getattr(opts, "hgr_class_metrics", False) else None
    hits = ops.new_hits(model.device)
    num_sample = 0
    out_str = ""
    with torch.no_grad():
        for i, data in enumerate(loader):
            imgs, targets = data["img"].to(device, non_blocking=True)[0], data["label"].to(device, non_blocking=True)[0]
            x = model.encode_image_normalized(imgs)
            _, idx = model.score_topk(None, targets, hits=hits, feats_normalized=x)   # main.py:135-147, fused
            num_sample += len(targets)
            if hier is not None:                                             # main.py:152: every row against targets[0]
                hier.update_rows(x, targets[:1].expand(len(targets)))
            if mist is not None:
                mist.update(idx, targets)
            if cls is not None:
                cls.update(idx, targets)
            if i % opts.print_freq == 0:
                out_str = _format(hits, num_sample, hier, mist, cls)
                print(out_str, flush=True)
    print("End of testing.")
    out_str = _format(hits, num_sample, hier, mist, cls)
    print(out_str, flush=True)
    if log:
        _log(opts, model, out_str)
    return out_str


def _test_splits(opts, model, device, splits, split_keys, loader, log):
    """``test`` for several split-file keys at once: one scoring pass per batch, one line per split."""
    if splits is None:
        raise ValueError("--hgr_eval_splits needs the split file's class lists (splits)")
    index = model.hierarchy.index
    se = SplitEval(model, {k: [index[c] for c in splits[k]] for k in split_keys},
                   hier=getattr(opts, "hgr_hier_metrics", True), mistakes=getattr(opts, "hgr_mistake_metrics", False),
                   class_metrics=getattr(opts, "hgr_class_metrics", False))
    with torch.no_grad():
        for i, data in enumerate(loader):
            imgs, targets = data["img"].to(device, non_blocking=True)[0], data["label"].to(device, non_blocking=True)[0]
            x = model.encode_image_normalized(imgs)
            se.update(x, targets, targets[:1].expand(len(targets)))        # TOR / POR: main.py:152, targets[0]
            if i % opts.print_freq == 0:
                print("\n" + "\n".join(se.lines()), flush=True)
    print("End of testing.")
    out_str = "\n" + "\n".join(se.lines())
    print(out_str, flush=True)
    if log:
        _log(opts, model, out_str)
    return out_str


def _log(opts, model, out_str):
    with open(model.save_path + "arugements.log", "a") as f:           # [sic] main.py:217
        f.writelines(out_str + "\n")
    with open("{}.txt".format(opts.weights), "a") as f:                # main.py:219-222
        method = "{},{},{}:".format(opts.weights, opts.out_ratio, opts.in_ratio)
        f.writelines(method + "\n" + out_str + "\n")


def _format(hits, num_sample, hier, mist=None, cls=None):
    out_str, _ = count_acc(dict(zip(HIT_CUTS, hits.tolist())), num_sample)
    out_str = "\n" + out_str
    if hier is not None:
        out_str += hier_line(*hier.ratios(num_sample))
    if mist is not None:
        out_str += mistake_line(mist.summary())
    if cls is not None:
        out_str += class_line(cls.summary())
    return out_str
