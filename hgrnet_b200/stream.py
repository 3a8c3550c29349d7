"""Streaming eval step with static buffers, replayed as CUDA graphs on a few round-robin streams.

The reference's eval loop (main.py:131-148) launches ~10 small torch ops per batch from Python;
at B200 speeds one batch of the fused head is ~20 us of GPU time, less than the CPU cost of
issuing it, and a large part of those 20 us is per-kernel fixed latency (launch, TMEM/barrier
set-up, first HBM touch, grid tail).  ``EvalStream`` removes both from the per-batch path: for a
fixed batch shape it owns pinned host staging buffers (the place a ``pin_memory=True`` loader
writes into, dataset/imagenet_group_test.py:83), device buffers and one captured CUDA graph per
slot that does

    H2D(features, labels) -> row-normalise (kernel 1) -> fused logits/top-K/Hit@k (kernel 2 + merge)
    -> D2H(hit counters)

A step is one ``cudaGraphLaunch``.  Consecutive slots are replayed on different streams (batches
are independent), so the copy of batch i+1 and the small kernels of neighbouring batches overlap
the GEMM of batch i and CTAs of the next GEMM start as soon as SMs drain.  Results (top-K values /
node ids) stay in the slot's device buffers; the Hit@{1,2,5,10,20} counters accumulate on the
device (atomics commute) and are mirrored to pinned host memory every step.

With ``hier`` (an ``evaluate.HierMetrics``) each graph also runs the hierarchical metrics TOR / POR
(main.py:143,152-191) on the slot's per-row labels after the scoring call
(``ops.hier_metrics_fused_rows``: per-level arg-max in the epilogue of a GEMM against the level-sorted train bank, then
per-row chain matching).  Its per-chain-length counters share one device buffer with the hit counters, so a step still
makes one D2H copy.  The level-sorted train bank, like ``bank``, is taken when the stream is built: after a bank
refresh, build a new stream.

With ``splits`` (an ``evaluate.SplitEval``) each graph scores the batch against all of the SplitEval's test splits in
one pass instead of against ``bank`` (``ops.score_topk_splits`` over the union bank, plus the per-split TOR / POR when
the SplitEval has them): one line per split, same graph shape, and the per-split counters sit in the same device buffer
as the others, so a step still makes one D2H copy (``split_hit_counts`` / ``split_ratios``).  The union bank too is taken
when the stream is built.

With ``mistakes`` (an ``evaluate.MistakeMetrics``) each graph also counts the mistake severity and LCA distance@k of
the slot's top-K lists against its per-row labels (``ops.hier_mistakes``, one warp per row), one counter set per split
with ``splits``.  These counters too sit in the one device buffer (``mistake_summary`` / ``split_mistake_summary``).

With ``classes`` (an ``evaluate.ClassHits``) each graph also counts Hit@k per class of the slot's top-K lists against
its per-row labels (``ops.class_hits``, one thread per row), one table per split with ``splits``.  The table
(``class_counts``, 1 MB per set at 21,841 nodes) is a device buffer of its own: the per-step D2H copy stays the few KB
of ``counters``, and the table is read only at readout (``class_table`` / ``class_summary`` / ``split_class_summary``).

With two or more streams, neighbouring batches' scoring kernels run side by side, so each graph's scoring call asks for
the grid share the library recommends for the batch shape (``ops.score_topk_grid_share``): on short streams (cfg 2:
B = 512 against 21,841 classes) each batch takes half the CTA pairs and runs twice as many columns per worker, instead
of every batch paying the kernel's fixed costs on every SM.  ``grid_share`` / ``plan()`` report what the slots run;
``concurrent=`` overrides the share.  ``splits`` keeps the whole grid.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops
from .evaluate import EvalCounters


class EvalStream:
    def __init__(self, bank: torch.Tensor, col_id: Optional[torch.Tensor] = None, id_base: int = 0, *, batch: int,
                 feat_dtype=torch.float32, K: int = 20, slots: int = 4, streams: int = 2, banks=None,
                 host_io: bool = True, hier=None, splits=None, mistakes=None, classes=None,
                 concurrent: Optional[int] = None):
        """``bank`` [C, D] bf16 on the device.  ``banks``: optional list of bank tensors to rotate over per slot
        (benchmarks use it to keep the working set larger than L2).  ``host_io=False`` skips the H2D / D2H nodes
        (features are then written straight into ``dev_feats`` / ``dev_labels``).  ``hier``: optional
        ``evaluate.HierMetrics`` of the model; when given, every step also counts TOR / POR (``hier_ratios``).  Labels
        are node ids; a label outside the hierarchy (e.g. -1 padding) is counted by neither metric.  ``splits``: optional
        ``evaluate.SplitEval``; every step then scores against its splits instead of ``bank`` (``val`` / ``idx`` are
        ``[S, B, K]``, ``hit_counts`` stays zero, ``split_hit_counts`` / ``split_ratios`` give the per-split results).
        ``mistakes``: optional ``evaluate.MistakeMetrics`` of the model (its chain table); every step then also counts the
        mistake severity and LCA distance@k of the slot's lists (``mistake_summary`` / ``split_mistake_summary``).
        ``classes``: optional ``evaluate.ClassHits`` of the model; every step then also counts the slot's Hit@k per class
        (``class_table`` / ``class_summary`` / ``split_class_summary``).  ``concurrent``: the grid share of every
        slot's scoring call (``ops.score_topk(grid_share=...)``, 1 = the whole grid); by default the library's
        recommendation for the batch shape with two or more streams, else 1."""
        self.device = bank.device
        self.K = K
        self.B = batch
        D = bank.shape[1]
        self.banks = list(banks) if banks is not None else [bank]
        self.col_id, self.id_base = col_id, id_base
        self.slots = slots
        self.host_io = host_io
        # features and labels of a slot share ONE staging buffer on each side, so a batch is a single DMA (a second,
        # 2 KB copy costs a descriptor's fixed latency on the same copy engine that carries the 2 MB of features)
        fbytes = batch * D * torch.empty((), dtype=feat_dtype).element_size()
        nbytes = fbytes + batch * 4

        def views(pack):
            return pack[:fbytes].view(feat_dtype).view(batch, D), pack[fbytes:].view(torch.int32)

        self.dev_pack = [torch.zeros(nbytes, dtype=torch.uint8, device=self.device) for _ in range(slots)]
        self.dev_feats, self.dev_labels = map(list, zip(*[views(p) for p in self.dev_pack]))
        # every counter of the stream in one device buffer (evaluate.EvalCounters): one D2H copy per step
        if hier is not None and splits is not None:
            raise ValueError("splits and hier together: the splits' TOR / POR come with the SplitEval's hier")
        self.hier = hier
        self.splits = splits
        self.mistakes = mistakes
        self._split_args = splits.score_args() if splits is not None else None
        hier = hier if splits is None else splits.hier
        self._hier_args = hier.rows_args() if hier is not None else None
        self._mistake_args = mistakes.args() if mistakes is not None else None
        self._node_splits = None if splits is None else splits.node_splits
        self.tally = EvalCounters(self.device, n_splits=0 if splits is None else splits.S, hier=hier is not None,
                                  mistakes=mistakes is not None, K=K, read=self._read_counters,
                                  classes=0 if classes is None else classes.n_nodes)
        self.counters, self.hits = self.tally.counters, self.tally.hits
        self.split_counts, self.hier_counts = self.tally.split_counts, self.tally.hier_counts
        self.mistake_counts = self.tally.mistake_counts
        self.class_counts = self.tally.class_counts
        if host_io:
            self.host_pack = [torch.zeros(nbytes, dtype=torch.uint8).pin_memory() for _ in range(slots)]
            self.host_feats, self.host_labels = map(list, zip(*[views(p) for p in self.host_pack]))
            self.host_counters = torch.zeros(self.counters.numel(), dtype=torch.int64).pin_memory()
            self.host_hits = self.host_counters[:ops.HGR_NUM_HITS]
        self.val = [None] * slots
        self.idx = [None] * slots
        self.streams = [torch.cuda.Stream(device=self.device) for _ in range(max(1, min(streams, slots)))]
        if splits is not None and concurrent not in (None, 1):
            raise ValueError("concurrent: the grid share applies to the single-bank scoring call, not to splits")
        if concurrent is not None:
            self.grid_share = int(concurrent)
        elif splits is None and len(self.streams) >= 2:
            self.grid_share = ops.score_topk_grid_share(batch, bank.shape[0], D, K)
        else:
            self.grid_share = 1
        self.graphs = []
        self.num_samples = 0
        self._capture()

    def _stream_of(self, slot: int):
        return self.streams[slot % len(self.streams)]

    def _body(self, s: int):
        if self.host_io:
            self.dev_pack[s].copy_(self.host_pack[s], non_blocking=True)
        x = ops.normalize_rows(self.dev_feats[s])                                    # clip_tree.py:330
        if self._split_args is None:                                                 # clip_tree.py:331 + main.py:136-147
            self.val[s], self.idx[s] = ops.score_topk(x, self.banks[s % len(self.banks)], col_id=self.col_id,
                                                      id_base=self.id_base, targets=self.dev_labels[s], K=self.K,
                                                      hits=self.hits, grid_share=self.grid_share)
        else:                                                                        # the same, once per test split
            self.val[s], self.idx[s] = ops.score_topk_splits(x, targets=self.dev_labels[s], counts=self.split_counts,
                                                             **self._split_args)
        if self._hier_args is not None:                                              # main.py:143,152-191
            ops.hier_metrics_fused_rows(x, targets=self.dev_labels[s], counts=self.hier_counts,
                                        node_splits=self._node_splits, **self._hier_args)
        if self._mistake_args is not None:                                           # main.py:135-148, hierarchy distance
            ops.hier_mistakes(self.idx[s], self.dev_labels[s], counts=self.mistake_counts, node_splits=self._node_splits,
                              **self._mistake_args)
        if self.class_counts is not None:                                            # main.py:135-148, per class
            ops.class_hits(self.idx[s], self.dev_labels[s], self.class_counts, node_splits=self._node_splits)
        if self.host_io:
            self.host_counters.copy_(self.counters, non_blocking=True)

    def _capture(self):
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(cur)
        # a slot is always captured and replayed on the same stream: the kernel workspace is per stream
        for s in range(self.slots):
            with torch.cuda.stream(self._stream_of(s)):
                self._body(s)                             # warm-up: workspace allocation, lazy module loading
        for st in self.streams:
            st.synchronize()
        self.tally.zero_()
        torch.cuda.synchronize(self.device)
        for s in range(self.slots):
            st = self._stream_of(s)
            with torch.cuda.stream(st):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=st):
                    self._body(s)
                self.graphs.append(g)
        torch.cuda.synchronize(self.device)

    def plan(self) -> dict:
        """What every slot's scoring call runs (``ops.score_topk_plan`` at ``grid_share``), with ``grid_share``.  Needs
        no ``splits``."""
        if self.splits is not None:
            raise ValueError("plan(): the slots score against splits (ops.score_topk_splits)")
        C, D = self.banks[0].shape
        return dict(ops.score_topk_plan(self.B, C, D, self.K, grid_share=self.grid_share), grid_share=self.grid_share)

    # ------------------------------------------------------------------ per-batch API
    def begin(self):
        """Order the worker streams after everything already queued on the caller's current stream."""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(cur)

    def step(self, slot: int):
        """Score the batch held in ``host_feats[slot]`` / ``host_labels[slot]`` (one graph launch; returns at once)."""
        with torch.cuda.stream(self._stream_of(slot)):
            self.graphs[slot].replay()
        self.num_samples += self.B

    def end(self):
        """Make the caller's current stream wait for all steps issued so far."""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def synchronize(self):
        for st in self.streams:
            st.synchronize()

    # ------------------------------------------------------------------ readout (evaluate.EvalCounters)
    def _read_counters(self, counters):
        # the per-step D2H copies of several streams land in the same bytes in no particular order: read the device
        # counters once every stream is idle
        self.synchronize()
        return counters

    def hit_counts(self):
        """Hit@{1,2,5,10,20} so far (synchronises)."""
        return self.tally.hit_counts()

    def hier_ratios(self):
        """``(hit_ratio, path_ratio, point_ratio)`` in percent -- the TOR / POR of the reference's ``test()`` line -- over
        the rows scored so far whose label lies in the hierarchy (synchronises).  Needs ``hier``."""
        return self.tally.hier_ratios()

    def split_hit_counts(self):
        """Per split ``[Hit@1, @2, @5, @10, @20, rows]`` so far, in the order of ``splits.names`` (synchronises)."""
        return self.tally.split_hit_counts()

    def split_ratios(self):
        """Per split ``(hit_ratio, path_ratio, point_ratio)`` in percent over the rows whose label is in the split
        (synchronises).  Needs ``splits`` with TOR / POR."""
        return self.tally.split_ratios()

    def mistake_summary(self):
        """``evaluate.mistake_summary`` of the rows scored so far (synchronises).  Needs ``mistakes`` without
        ``splits``."""
        return self.tally.mistake_summary()

    def split_mistake_summary(self):
        """Per split ``evaluate.mistake_summary`` over the rows whose label is in the split, in the order of
        ``splits.names`` (synchronises).  Needs ``mistakes`` and ``splits``."""
        return self.tally.split_mistake_summary()

    def class_table(self) -> torch.Tensor:
        """The per-class table so far, host int64 ``[n_nodes, 6]`` (``[S, n_nodes, 6]`` with ``splits``): per class
        ``[Hit@1, @2, @5, @10, @20, rows]`` (synchronises).  Needs ``classes``."""
        return self.tally.class_table()

    def class_summary(self):
        """``evaluate.class_summary`` of the rows scored so far (synchronises).  Needs ``classes`` without ``splits``."""
        return self.tally.class_summary()

    def split_class_summary(self):
        """Per split ``evaluate.class_summary`` over the rows whose label is in the split, in the order of
        ``splits.names`` (synchronises).  Needs ``classes`` and ``splits``."""
        return self.tally.split_class_summary()
