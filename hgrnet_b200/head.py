"""``tree_model``: drop-in for the reference's hierarchy-aware CLIP wrapper (model/clip_tree.py).

Same constructor arguments, methods and attributes as the reference class as used by its
``main.py`` (SURVEY.md section 8b); the hot path behind them runs in ``libhgr_b200.so``:

* ``update_classifier``  -> kernel (1) ``hgr_aggregate_normalize``   (clip_tree.py:318-325)
* ``forward``            -> kernel (1) + ``hgr_logits_dense``        (clip_tree.py:328-333)
* ``score_topk`` (NEW)   -> kernel (1) + kernel (2) ``hgr_score_topk`` fused logits/top-20/Hit@k
                            (clip_tree.py:330-331 + main.py:136-147), no [B,N] matrix
* ``train_batch``        -> kernel (1) + ``hgr_logits_dense`` + kernel (3) ``hgr_masked_ce``
                            (clip_tree.py:222-316), all (k,m) iterations in one launch

The CLIP encoders stay upstream torch modules (``clip_model.encode_image`` / ``encode_text``);
only their output contract matters.  There is no CPU path: tensors must live on a CUDA device.
"""
from __future__ import annotations

import copy
import os
import random
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .hierarchy import Hierarchy
from .levels import iteration_weights_grad_np, iteration_weights_np, layer_weight_init, level_weights
from .sampling import (contra_brothers, contra_random, contra_topk, contra_topk_many, hierarchical_schedule, om_plan, om_schedule,
                       sample_stream)

TEMPLATE_SIMPLE = "a photo of a {}."  # data/templates.py:98-100 (TEMPLATES_SIMPLE[0], hard-wired at clip_tree.py:52)


def _default_node_names(nodes: Sequence[str]) -> List[str]:
    """Prompt names as in clip_tree.py:53-58 (WordNet lemma of the wnid); falls back to the wnid."""
    try:
        from nltk.corpus import wordnet as wn  # optional upstream dependency
    except Exception:  # pragma: no cover - nltk is not part of this image
        wn = None
    names = []
    for node in nodes:
        name = node
        if wn is not None:
            try:
                name = wn.synset_from_pos_and_offset("n", int(node[1:])).name().split(".")[0].replace("_", " ")
            except Exception:
                name = node
        names.append(TEMPLATE_SIMPLE.format(name))
    return names


class tree_model(nn.Module):
    def __init__(self, opts, candidates_train, candidates_test, clip_model: Optional[nn.Module] = None,
                 hierarchy: Optional[Hierarchy] = None, node_tokens: Optional[torch.Tensor] = None,
                 tokenizer=None):
        super().__init__()
        self.opts = opts
        self.device = torch.device("cuda:%d" % opts.device) if isinstance(opts.device, int) else torch.device(opts.device)
        self.save_path = "{}/{}/{}_{}_{}/".format(opts.folder, opts.exp_name, opts.weights, opts.out_ratio, opts.in_ratio)
        self.file_path = self.save_path + "clip_{}".format(opts.from_epoch)
        if not os.path.exists(self.save_path):
            os.makedirs(self.save_path)

        # semantic structure (utils.gen_tree, utils.py:39-72)
        self.hierarchy = hierarchy if hierarchy is not None else Hierarchy.from_json(opts.graph_path)
        self.p2c, self.c2p, self.d2n, self.nodes, self.start_up = self.hierarchy.as_tuple()
        self.nodes_id = list(range(len(self.nodes)))

        # upstream encoders
        if clip_model is None:
            try:
                import clip  # the upstream OpenAI package / the reference's vendored copy on PYTHONPATH
            except ImportError as e:
                raise ImportError("pass clip_model=... or put an OpenAI-CLIP compatible `clip` package on "
                                  "PYTHONPATH: the encoders are upstream producers, not part of hgrnet_b200") from e
            clip_model, _ = clip.load(name=opts.arch, device=self.device, download_root="pretrained")
            if tokenizer is None:
                tokenizer = clip.tokenize
        self.clip_model = clip_model
        if getattr(opts, "fetch", False):
            self.clip_model.load_state_dict(torch.load(opts.fetch_path))
        if getattr(opts, "load", False):
            path = self.file_path if opts.load_path == "none" else opts.load_path
            self.clip_model.load_state_dict(torch.load(path))
            print("successfully loaded")
        self.clip_model.eval()
        for params in self.clip_model.parameters():
            params.requires_grad_(True)

        # prompts -> tokens (clip_tree.py:52-60)
        if node_tokens is None:
            if tokenizer is None:
                raise ValueError("node_tokens or tokenizer required when clip_model is supplied")
            with torch.no_grad():
                node_tokens = tokenizer(_default_node_names(self.nodes))
        self.node_tokens = node_tokens.to(self.device)

        # misc (clip_tree.py:63-68)
        self.resolution = getattr(getattr(self.clip_model, "visual", None), "input_resolution", 224)
        self.candidates_train = candidates_train
        self.candidates_test = candidates_test
        index = self.hierarchy.index
        self.train_index = torch.tensor([index[c] for c in candidates_train], dtype=torch.long, device=self.device)
        self.test_index = torch.tensor([index[c] for c in candidates_test], dtype=torch.long, device=self.device)
        self._train_ids_host = [index[c] for c in candidates_train]
        # Row order of the test-class bank (kernel 2's B operand).  The reference's `nodes` order is graph order --
        # siblings adjacent and similar -- so an image's top-20 concentrate in a few adjacent bank rows, the one
        # case the narrow speculative lists of the scoring kernel are slow for (exact, but repaired on the CUDA
        # cores).  A fixed pseudo-random permutation of the bank rows makes their order independent of the hierarchy;
        # `_test_index_i32` (the kernel's col_id) maps bank rows back to node ids, so nothing else changes -- except
        # that exact ties resolve by permuted row instead of by test_index position (torch.topk's tie order is
        # unspecified anyway, main.py:138).  `opts.hgr_permute_bank = False` keeps test_index order.
        C = self.test_index.numel()
        if getattr(opts, "hgr_permute_bank", True) and C > 1:
            perm = torch.randperm(C, generator=torch.Generator().manual_seed(0x48475221)).to(self.device)
        else:
            perm = torch.arange(C, device=self.device)
        self._bank_order = self.test_index[perm]                         # node id of bank_test row j
        self._test_index_i32 = self._bank_order.to(torch.int32)
        self._bank_dst = torch.full((len(self.nodes),), -1, dtype=torch.int32, device=self.device)
        self._bank_dst[self._bank_order] = torch.arange(C, dtype=torch.int32, device=self.device)   # node -> bank row
        self.max_depth = max(self.d2n.keys())

        if self.opts.weights == "adaptive":
            # The reference builds a NON-leaf tensor here (clip_tree.py:74, SURVEY.md section 0), which
            # makes its own optimizer2 unusable.  Same values, but a real Parameter named "layer_weight"
            # so that main.py's filters (`name != "layer_weight"`, SGD([model.layer_weight])) work.
            self.layer_weight = nn.Parameter(layer_weight_init(self.d2n, self.opts.scale).to(self.device))

        self.zsl_weights: Optional[torch.Tensor] = None   # [N, D] bf16 class bank
        self.bank_test: Optional[torch.Tensor] = None     # [C, D] bf16 rows of test_index (in `_bank_order`)
        self.bank_train: Optional[torch.Tensor] = None    # [M, D] bf16 rows of train_index
        self._rng = random  # Python's global RNG, as the reference (clip_tree.py:82,134,189)
        self._contra_cache = {}  # depth window -> candidate set (sampling.contra_topk)

    # ------------------------------------------------------------------ checkpoint
    def save(self, opts, epoch):
        """clip_tree.py:76-78."""
        torch.save(self.clip_model.state_dict(), self.save_path + "clip_{}".format(epoch))

    # ------------------------------------------------------------------ sampling / weights
    def _contra_ids(self, method, target, depth=None, parents=None, rng=None):
        rng = self._rng if rng is None else rng       # `rng`: Python's global generator or a SampleStream over it
        if method == "topk":
            return contra_topk(self.d2n, target, depth, parents, self.opts.k, self.opts.num_compare, rng,
                               cache=self._contra_cache)
        if method == "random":
            return contra_random(self._train_ids_host, target, self.opts.num_compare, rng)
        if method == "brothers":
            return contra_brothers(self.p2c, self.start_up, target, depth, parents, self.opts.num_compare, rng)
        raise NotImplementedError(
            "sample_strategy %r: the reference's 'simi'/'near_simi' branches (clip_tree.py:91-114,143-178) mix "
            "python lists with tensors and cannot run as published; supported: topk, random, brothers" % method)

    def get_contra(self, method, target, batch_size, depth=None, parents=None):
        """clip_tree.py:80-196 -> ``(compare_idx LongTensor[n], labels LongTensor[B])`` on the device."""
        ids, pos = self._contra_ids(method, target, depth, parents)
        compare_idx = torch.tensor(ids, device=self.device)
        return compare_idx, torch.full((batch_size,), pos, dtype=torch.long, device=self.device)

    def _layer_weight_host(self):
        lw = getattr(self, "layer_weight", None)
        return None if lw is None else lw.detach().float().cpu()

    def get_weights(self, method, max_depth=None):
        """clip_tree.py:198-219 -> fp32 tensor [max_depth] on the device."""
        lw = getattr(self, "layer_weight", None)
        w = level_weights(method, max_depth, lw)
        return w.to(self.device)

    # ------------------------------------------------------------------ class bank
    def _bank_csr(self):
        """CSR of the hierarchy-aggregated bank (north_star's extension; SURVEY section 0: the reference's own bank is the
        identity CSR).  `opts.hgr_bank`: "node" (default, = reference), "chain" -- row c aggregates the last
        ceil(out_ratio * len) nodes of c2p[c] + [c], deepest first, with the `--weights` level weights (the node set
        and weights the OM loop uses, clip_tree.py:232-237 / :198-219) -- or "family": the chain plus the direct
        children of c, which share a total weight of `in_ratio` (the descendant side)."""
        mode = getattr(self.opts, "hgr_bank", "node")
        if mode == "node":
            return None
        if mode not in ("chain", "family"):
            raise ValueError("opts.hgr_bank must be node, chain or family, got %r" % (mode,))
        lw = self._layer_weight_host()
        rp, col, w = self.hierarchy.chain_csr(self.opts.out_ratio,
                                              lambda n: level_weights(self.opts.weights, n, lw).numpy(),
                                              include_children=mode == "family", child_weight=float(self.opts.in_ratio))
        to = lambda a: torch.from_numpy(a).to(self.device)
        return to(rp), to(col), to(w)

    def update_classifier(self, chunk: int = 4096):
        """clip_tree.py:318-325.  The reference encodes the prompts in two halves, concatenates and normalises.
        Here every chunk of text features is normalised by kernel (1) STRAIGHT INTO its rows of the bf16 all-node bank
        and, in the same pass, into its (permuted) rows of the test-class bank (`hgr_normalize_rows_dual`): no
        concatenated copy of the text table, no second read.  With `--hgr_bank chain` the rows are hierarchy-aggregated
        (CSR over ancestors), which needs the whole text table first."""
        with torch.no_grad():
            N = len(self.nodes)
            csr = self._bank_csr()
            if csr is None:
                zsl = bank = None
                for s in range(0, N, chunk):
                    feats = self.clip_model.encode_text(self.node_tokens[s:s + chunk])
                    if zsl is None:
                        D = feats.shape[1]
                        zsl = torch.empty((N, D), dtype=torch.bfloat16, device=self.device)
                        bank = torch.empty((self._bank_order.numel(), D), dtype=torch.bfloat16, device=self.device)
                    e = s + feats.shape[0]
                    ops.normalize_rows_dual(feats, zsl[s:e], self._bank_dst[s:e], bank)
                self.zsl_weights, self.bank_test = zsl, bank
                self.bank_train = zsl.index_select(0, self.train_index)      # TOR / POR columns (evaluate.HierMetrics)
            else:
                text = None
                for s in range(0, N, chunk):
                    feats = self.clip_model.encode_text(self.node_tokens[s:s + chunk])
                    if text is None:
                        text = torch.empty((N, feats.shape[1]), dtype=feats.dtype, device=self.device)
                    text[s:s + feats.shape[0]] = feats
                rp, col, w = csr
                self.zsl_weights = ops.aggregate_normalize(text, rp, col, w)
                self.bank_test = ops.aggregate_normalize(text, rp, col, w, row_map=self._test_index_i32)
                self.bank_train = self.zsl_weights.index_select(0, self.train_index)

    # ------------------------------------------------------------------ eval
    def encode_image_normalized(self, inputs):
        feats = self.clip_model.encode_image(inputs)
        return ops.normalize_rows(feats.detach())

    def forward(self, inputs, targets=None):
        """clip_tree.py:328-333: cosine logits [B, N] (fp32) for ALL nodes."""
        x = self.encode_image_normalized(inputs)
        return ops.logits_dense(x, self.zsl_weights)

    def score_topk(self, inputs, targets, hits: Optional[torch.Tensor] = None, K: int = 20, feats_normalized=None):
        """Fused replacement of ``model(imgs)`` + main.py:136-147.

        Returns ``(val [B,K], idx [B,K] node ids)`` and accumulates Hit@{1,2,5,10,20} into ``hits``.
        """
        x = feats_normalized if feats_normalized is not None else self.encode_image_normalized(inputs)
        t = targets.to(torch.int32) if targets is not None else None
        return ops.score_topk(x, self.bank_test, col_id=self._test_index_i32, targets=t, K=K, hits=hits)

    def make_eval_stream(self, batch: int, slots: int = 4, streams: int = 2, feat_dtype=torch.float32, K: int = 20,
                         banks=None, host_io: bool = True, hier_metrics: bool = False, eval_splits=None,
                         mistake_metrics: bool = False, class_metrics: bool = False, concurrent=None):
        """CUDA-graph replayed eval step over pre-computed image features (hgrnet_b200.stream.EvalStream).

        ``hier_metrics=True`` adds TOR / POR (``EvalStream.hier_ratios``), every row scored against its own label.  The
        stream keeps the device pointers of ``bank_test`` and of the level-sorted ``bank_train`` taken now: after
        ``update_classifier`` refreshes the banks, build a new stream.

        ``eval_splits`` (``{name: node ids}``, at most 8 splits): every step scores against all of these test splits
        in one pass instead of against ``bank_test`` (``EvalStream.split_hit_counts``; with ``hier_metrics`` also the
        per-split TOR / POR, ``EvalStream.split_ratios``).

        ``mistake_metrics=True`` adds the mistake severity and LCA distance@k of every row's top-K against its own label
        (``EvalStream.mistake_summary``, per split ``EvalStream.split_mistake_summary``).

        ``class_metrics=True`` adds the Hit@k of every class, every row counted toward its own label
        (``EvalStream.class_table``; class-averaged: ``EvalStream.class_summary``, per split
        ``EvalStream.split_class_summary``).

        ``concurrent``: grid share of the slots' scoring calls (``EvalStream``'s ``concurrent``; default: the library's
        recommendation for the batch shape)."""
        from .stream import EvalStream
        hier = splits = mistakes = classes = None
        if class_metrics:
            from .evaluate import ClassHits
            classes = ClassHits(self, K=K)
        if mistake_metrics:
            from .evaluate import MistakeMetrics
            mistakes = MistakeMetrics(self, K=K)
        if eval_splits is not None:
            from .evaluate import SplitEval
            splits = SplitEval(self, eval_splits, hier=hier_metrics, K=K)
        elif hier_metrics:
            from .evaluate import HierMetrics
            hier = HierMetrics(self)
        return EvalStream(self.bank_test, col_id=self._test_index_i32, batch=batch, feat_dtype=feat_dtype, K=K,
                          slots=slots, streams=streams, banks=banks, host_io=host_io, hier=hier, splits=splits,
                          mistakes=mistakes, classes=classes, concurrent=concurrent)

    # ------------------------------------------------------------------ training step
    def _schedule(self, training_method, target):
        """Host-side expansion of the loop nest into T (anchor, depth, chain) requests and weight recipes."""
        if training_method not in ("OM", "hierarchical"):
            raise NotImplementedError("training_method %r (the reference implements OM and hierarchical)" % training_method)
        if training_method == "OM":
            weighting = self.opts.weighting                                          # clip_tree.py:265-273
            m_in = "equal" if weighting == "out" else self.opts.weights
            m_out = "equal" if weighting == "in" else self.opts.weights
            sched = om_schedule(self.c2p, target, self.opts.out_ratio, self.opts.in_ratio)
            requests = [(p_out, depth, parents_in) for (_, _, p_out, depth, parents_in, _, _) in sched]
            recipes = [((m_in, n_in, m_loop), (m_out, n_out, k_loop)) for (k_loop, m_loop, _, _, _, n_out, n_in) in sched]
        else:
            sched = hierarchical_schedule(self.c2p, target)
            requests = [(t_in, depth, parents) for (_, t_in, depth, parents, _) in sched]
            recipes = [((self.opts.weights, n_lvl, j),) for (j, _, _, _, n_lvl) in sched]      # clip_tree.py:304-305
        return requests, recipes

    def _plan_sets(self, requests, sample_strategy):
        """The T sampled class sets of a step as ``(set_ptr, set_col, label_pos, union)`` int32 numpy arrays: offsets,
        columns of the union, position of the anchor in every set, node ids of the union (ascending).  Every
        `random.sample` of the step runs on one SampleStream: same draws and same generator state afterwards as the
        reference's per-iteration calls (clip_tree.py:134); for `topk` the whole plan is one call of the library's host
        helper (`hgr_om_plan`)."""
        T = len(requests)
        with sample_stream(self._rng) as rng:
            if sample_strategy == "topk":
                planned = om_plan(self.d2n, requests, self.opts.k, self.opts.num_compare, rng, len(self.nodes),
                                  cache=self._contra_cache)
                if planned is not None:
                    return planned
                picked = contra_topk_many(self.d2n, requests, self.opts.k, self.opts.num_compare, rng,
                                          cache=self._contra_cache)
            else:
                picked = [self._contra_ids(sample_strategy, t, depth, parents, rng) for (t, depth, parents) in requests]
        # numpy path (other strategies / no library): union of the sampled classes, every set as columns of it
        lens = np.fromiter((len(ids) for ids, _ in picked), dtype=np.int64, count=T)
        cat = np.concatenate([np.asarray(ids, dtype=np.int64) for ids, _ in picked])
        union, inv = np.unique(cat, return_inverse=True)
        set_ptr = np.zeros(T + 1, dtype=np.int32)
        np.cumsum(lens, out=set_ptr[1:])
        return (set_ptr, inv.astype(np.int32), np.asarray([p for _, p in picked], np.int32), union.astype(np.int32))

    def train_batch(self, inputs, targets, training_method, sample_strategy):
        """clip_tree.py:222-316.  Returns the python-float loss sum; gradients are accumulated on the
        encoder parameters, ``logit_scale`` and ``layer_weight`` as a side effect (no zero_grad, as the
        reference)."""
        img_feats = self.clip_model.encode_image(inputs)
        x, x_norm = ops.normalize_rows(img_feats.detach(), return_norm=True)          # :225
        target = int(targets[0].item())                                                # :228 (single-label batch)
        B = x.shape[0]

        requests, recipes = self._schedule(training_method, target)
        T = len(requests)
        set_ptr, set_col, label_pos, union = self._plan_sets(requests, sample_strategy)
        lw_host = self._layer_weight_host()
        lw_param = getattr(self, "layer_weight", None)
        want_lw_grad = lw_param is not None and lw_param.requires_grad and self.opts.weights == "adaptive"
        # w_t = product of the level weights the recipe of iteration t names (clip_tree.py:265-273, :304-305), in numpy
        # (levels.iteration_weights_np); d loss / d layer_weight follows analytically at the end of the step
        lw_np = None if lw_host is None else lw_host.numpy()
        weight_np, w_ctx = iteration_weights_np(recipes, lw_np)
        # ONE host->device copy for everything the step's kernels read: offsets, columns, label positions, weights
        # (as raw fp32 bits) and the union ids
        n_col = int(set_col.shape[0])
        pack = np.concatenate([set_ptr, set_col, label_pos, weight_np.view(np.int32), union])
        meta = torch.from_numpy(pack).to(self.device, non_blocking=True)
        o1, o2, o3, o4 = T + 1, T + 1 + n_col, 2 * T + 1 + n_col, 3 * T + 1 + n_col
        d_set_ptr, d_set_col, d_label = meta[:o1], meta[o1:o2], meta[o2:o3]
        d_weight = meta[o3:o4].view(torch.float32)
        union_t = meta[o4:].long()

        # one encoder call for the union instead of T calls (:261); rows are independent in eval mode
        text_raw = self.clip_model.encode_text(self.node_tokens[union_t])
        tn, t_norm = ops.normalize_rows(text_raw.detach(), return_norm=True)          # :262
        scale = float(self.clip_model.logit_scale.detach().exp().item())
        logits = ops.logits_dense(x, tn, scale=scale)                                  # :263
        loss_t, dlogits = ops.masked_ce(logits, d_set_ptr, d_set_col, d_label, d_weight)   # :275-276

        # backward of logits = scale * x @ tn^T and of the two row normalisations: both gradient GEMMs on the tcgen05
        # kernel, normalise-backward and d(logit_scale) in the same library call (csrc/om_backward.cu)
        d_ls = torch.zeros(1, dtype=torch.float32, device=self.device)
        d_img_raw, d_text_raw = ops.om_backward(dlogits, logits, x, x_norm, tn, t_norm, scale, d_ls)
        d_log_scale = d_ls[0]
        ls = self.clip_model.logit_scale
        if ls.requires_grad:
            g = d_log_scale.to(ls.dtype).reshape(ls.shape)
            ls.grad = g if ls.grad is None else ls.grad + g
        # one pass of the autograd engine for both encoders (clip_tree.py:276 per iteration, :280)
        roots = [(t, g.to(t.dtype)) for t, g in ((text_raw, d_text_raw), (img_feats, d_img_raw)) if t.requires_grad]
        if roots:
            torch.autograd.backward([t for t, _ in roots], [g for _, g in roots])

        loss_host = loss_t.cpu()                                                        # the step's only result read-back
        if want_lw_grad:
            ce = loss_host.numpy() / weight_np                                          # d loss_t / d w_t = CE_t
            g = torch.from_numpy(iteration_weights_grad_np(w_ctx, ce, lw_np)).to(lw_param.device, lw_param.dtype)
            lw_param.grad = g if lw_param.grad is None else lw_param.grad + g
        self.last_losses = loss_host.tolist()
        return sum(self.last_losses)                                                    # :279
