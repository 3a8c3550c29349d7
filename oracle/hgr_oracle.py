"""fp32 CPU restatement of HGR-Net's hierarchical zero-shot scoring head.

TEST INFRASTRUCTURE ONLY -- the checker for ``hgrnet_b200``; never shipped, never on the
product path (see ``oracle/__init__.py``).

Every function restates, in plain torch-CPU fp32 / python, what the reference computes for
the hot path of SURVEY.md section 8 and cites the reference ``file:line`` it follows
(paths relative to the reference checkout).  Parity pin: the reference ships no tests or
golden vectors for this path (SURVEY.md section 4) -- "parity unpinned" by the reference's
own tests.  The pin used instead is the reference ITSELF: ``oracle/gen_golden.py`` imports
``/root/reference`` through ``oracle/ref_harness.py`` in the build container, runs the
unmodified ``tree_model`` / ``main.test`` code on seeded inputs and (a) asserts that this
restatement reproduces it, (b) freezes the outputs under ``tests/golden/``.

Precision rule (SURVEY.md section 8c): inputs are bf16-VALUED fp32 tensors, all arithmetic
is fp32 on CPU.  Never run this oracle in bf16/fp16.
"""
from __future__ import annotations

import copy
import math
import random as _random
from collections import OrderedDict, defaultdict, deque
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

ROOT = "fall11"  # utils.py:45,46,55 -- hard-wired root wnid of the edge list
TOPK = (1, 2, 5, 10, 20)  # main.py:120


# --------------------------------------------------------------------------- hierarchy
def gen_tree(edges: Sequence[Sequence[str]]):
    """Hierarchy index structures.  Follows utils.py:39-72 (``gen_tree``).

    * ``nodes``: graph-node insertion order of ``nx.DiGraph.add_edges_from`` (each edge adds
      its parent then its child if unseen), root removed (utils.py:42-45).
    * ``start_up``: children of the root (utils.py:46).
    * ``p2c[i]``: children ids in edge order (utils.py:48-51).
    * ``c2p[i]``: ids of the interior of one shortest root->i path (utils.py:53-56).  On a
      tree the path is unique.  On a DAG networkx's choice among equal-length paths is
      version dependent (SURVEY.md section 8c); this restatement takes the BFS-first parent.
    * ``d2n``: depth -> node ids, keys in order of first occurrence (utils.py:66-70).
    """
    succ: "OrderedDict[str, List[str]]" = OrderedDict()
    for u, v in edges:
        if u not in succ:
            succ[u] = []
        if v not in succ:
            succ[v] = []
        if v not in succ[u]:
            succ[u].append(v)
    nodes = [n for n in succ.keys() if n != ROOT]
    index = {n: i for i, n in enumerate(nodes)}
    start_up = [index[c] for c in succ[ROOT]]
    p2c = [[index[c] for c in succ[n]] for n in nodes]

    parent: Dict[str, Optional[str]] = {ROOT: None}
    queue = deque([ROOT])
    while queue:
        u = queue.popleft()
        for v in succ[u]:
            if v not in parent:
                parent[v] = u
                queue.append(v)
    c2p: List[List[int]] = []
    for n in nodes:
        chain = []
        p = parent[n]
        while p is not None and p != ROOT:
            chain.append(index[p])
            p = parent[p]
        c2p.append(chain[::-1])

    # utils.py:58-64 -- every consecutive pair of the chain must be a parent/child edge
    for i in range(len(nodes)):
        for a, b in zip(c2p[i][:-1], c2p[i][1:]):
            assert b in p2c[a]

    d2n: "defaultdict[int, List[int]]" = defaultdict(list)
    for i in range(len(nodes)):
        d2n[len(c2p[i])].append(i)
    return p2c, c2p, d2n, nodes, start_up


# --------------------------------------------------------------------------- level weights
def layer_weight_init(d2n, scale: float) -> torch.Tensor:
    """clip_tree.py:70-74: ``1/|level|`` in d2n *insertion* order, times ``--scale``."""
    num_layer = [len(d2n[layer]) for layer in d2n.keys()]
    return (1.0 / torch.tensor(num_layer)) * scale


def get_weights(method: str, n: int, layer_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """clip_tree.py:198-219 (``get_weights``), fp32 vector of length ``n``."""
    if method == "equal":
        return torch.ones(n) / n
    if method == "decreasing":
        w = torch.arange(start=n, end=0, step=-1)
        return w / w.sum()
    if method == "increasing":
        w = torch.arange(start=1, end=n + 1)
        return w / w.sum()
    if method == "adaptive":
        return F.softmax(100 ** layer_weight[:n], dim=0)
    if method == "nl_increasing":
        w = torch.arange(start=1, end=n + 1) ** 3
        return w / w.sum()
    if method == "nl_decreasing":
        w = torch.arange(start=n, end=0, step=-1) ** 3
        return w / w.sum()
    raise ValueError(method)


# --------------------------------------------------------------------------- sampling
def get_contra_topk(d2n, target: int, batch_size: int, depth: int, parents: Sequence[int],
                    k: int, num_compare: int, rng=_random) -> Tuple[List[int], List[int]]:
    """clip_tree.py:116-141 (``get_contra(method='topk')``).

    Candidates are every node at depths ``[max(min_depth, depth-k), depth-1]`` (plus depth 0
    itself when ``depth == 0``), minus the anchor chain ``parents``; sub-sampled to
    ``num_compare`` with ``random.sample``; the anchor is appended if absent.  Returns the
    id list and the label list (position of the anchor, repeated ``batch_size`` times).
    ``rng`` must expose ``sample`` (the ``random`` module or a ``random.Random``).
    """
    low = min(d2n.keys())
    if depth - k > low:
        low = depth - k
    candi: List[int] = []
    for d in range(low, depth):
        candi.extend(d2n[d])
    if depth == 0:
        candi.extend(d2n[depth])
    compare_idx = list(set(candi) - set(parents))
    if len(compare_idx) > num_compare:
        compare_idx = rng.sample(compare_idx, num_compare)
    if target not in compare_idx:
        compare_idx.append(target)
    label = compare_idx.index(target)
    return compare_idx, [label] * batch_size


def om_schedule(c2p, target: int, out_ratio: float, in_ratio: float):
    """Loop structure of the OM step, clip_tree.py:228-256.

    Yields ``(k_loop, m_loop, p_out, depth, parents_in, len_out_loop, len_in_loop)``.
    """
    parents = list(c2p[target]) + [target]
    k = math.ceil(out_ratio * len(parents))
    if k == 0:
        k = 1
    p_loop_out = parents[::-1][:k]
    sched = []
    for k_loop, p_out in enumerate(p_loop_out):
        parents_in = list(c2p[p_out]) + [p_out]
        m = math.ceil(in_ratio * len(parents_in))
        if m == 0:
            m = 1
        p_loop_in = parents_in[::-1][:m]
        for m_loop, p_in in enumerate(p_loop_in):
            depth = parents_in.index(p_in)
            sched.append((k_loop, m_loop, p_out, depth, parents_in, len(p_loop_out), len(p_loop_in)))
    return sched


# --------------------------------------------------------------------------- class bank
def normalize_rows(x: torch.Tensor) -> torch.Tensor:
    """``x / x.norm(dim=-1, keepdim=True)`` -- clip_tree.py:323 (bank), :330 (images)."""
    x = x.float()
    return x / x.norm(dim=-1, keepdim=True)


def aggregate_normalize(E: torch.Tensor, rowptr: Sequence[int], col: Sequence[int],
                        w: Sequence[float]) -> torch.Tensor:
    """``out[c] = normalize(sum_j w[c,j] * E[col[c,j]])``.

    Generalisation named by north_star; operator shape follows the DGP baseline's grouped
    adjacency aggregation + ``F.normalize`` (baseline/DGP/models/gcn_dense_att.py:31-46,
    :116).  With the identity CSR it is exactly ``update_classifier``'s normalise step
    (clip_tree.py:323) -- the only configuration with main-path reference parity.
    """
    E = E.float()
    rowptr_t = torch.as_tensor(rowptr, dtype=torch.long)
    col_t = torch.as_tensor(col, dtype=torch.long)
    w_t = torch.as_tensor(w, dtype=torch.float32)
    n = rowptr_t.numel() - 1
    row_of = torch.repeat_interleave(torch.arange(n), rowptr_t[1:] - rowptr_t[:-1])
    acc = torch.zeros(n, E.shape[1], dtype=torch.float32)
    acc.index_add_(0, row_of, E[col_t] * w_t[:, None])
    return acc / acc.norm(dim=-1, keepdim=True)


# --------------------------------------------------------------------------- eval head
def forward_logits(feats: torch.Tensor, bank: torch.Tensor) -> torch.Tensor:
    """clip_tree.py:330-331: row-normalise image feats, unscaled cosine logits vs bank."""
    feats = feats.float()
    feats = feats / feats.norm(dim=-1, keepdim=True)
    return feats @ bank.float().T


def eval_hits(logits: torch.Tensor, test_index: torch.Tensor, targets: torch.Tensor,
              topk: Sequence[int] = TOPK):
    """main.py:136-147: column-select, sorted top-20, map to node ids, cumulative Hit@k.

    Returns ``(pred [maxk,B] int64 node ids, vals [B,maxk] fp32, hits {k: int})``.
    """
    sel = logits[:, test_index]
    maxk = max(topk)
    vals, pred = sel.topk(maxk, 1, True, True)
    pred = test_index[pred].t()
    correct = pred.eq(targets.reshape(1, -1).expand_as(pred))
    hits = {k: int(correct[:k].reshape(-1).float().sum().item()) for k in topk}
    return pred, vals, hits


def count_acc(hits_dict, num_tot):
    """utils.py:135-146: ``Top@k(%):xx.xx, ...`` string and the accuracy dict."""
    parts = []
    acc = {}
    for key, value in hits_dict.items():
        acc[key] = value / num_tot * 100.0
        parts.append("Top@{}(%):{:.2f}".format(key, acc[key]))
    return ", ".join(parts) + ".", acc


def tor_por_winners(logits: torch.Tensor, train_index: torch.Tensor, c2p, d2n, n_nodes: int, target: int):
    """The arg-maxes behind ``tor_por`` (main.py:155-156,162-176): ``(top1 [B], dict_path [B, L])`` int64 node ids,
    the top-1 over ``train_index`` and, per node of the label's chain ``c2p[target] + [target]``, the top-1 over
    ``train_index`` after every column not at that node's depth is filled with -1."""
    B = logits.shape[0]
    parents = list(c2p[target]) + [target]
    L = len(parents)
    top1 = train_index[logits[:, train_index].topk(1, 1, True, True)[1]].squeeze(1)
    dict_path = torch.zeros(B, L, dtype=torch.long)
    for kk, p in enumerate(parents):
        level = len(c2p[p])
        same_l = list(d2n[level])
        if p not in same_l:
            same_l.append(p)
        rest = torch.tensor(sorted(set(range(n_nodes)) - set(same_l)), dtype=torch.long)
        lk = logits.clone().index_fill(1, rest, -1)[:, train_index]
        dict_path[:, kk] = train_index[lk.topk(1, 1, True, True)[1]].squeeze(1)
    return top1, dict_path


def tor_por(logits: torch.Tensor, train_index: torch.Tensor, c2p, d2n, n_nodes: int,
            target: int):
    """Hierarchical metrics of one single-label batch, main.py:143,152-191.

    Returns ``(tor_hits, path_add, point_add)``: the increments the reference adds to
    ``hits_all``, ``path_all`` and ``point_all`` for this batch.
    """
    B = logits.shape[0]
    parents = list(c2p[target]) + [target]
    L = len(parents)
    # TOR (main.py:143,155-160): top-1 over train_index matched against the whole chain
    # POR (main.py:162-176): per chain level, arg-max restricted to that level's nodes
    top1, dict_path = tor_por_winners(logits, train_index, c2p, d2n, n_nodes, target)
    tor_hits = float(top1[:, None].expand(B, L).eq(torch.tensor(parents).expand(B, L)).float().sum())
    # main.py:177-191
    path_add = 0.0
    edge = 0
    point = 0
    for i in range(B):
        if L - 1 == 0 and parents[0] == dict_path[i][0]:
            path_add += 1
        for j in range(L - 1):
            if parents[j] == dict_path[i][j]:
                point += 1
            if parents[j] == dict_path[i][j] and parents[j + 1] == dict_path[i][j + 1]:
                edge += 1
        if parents[L - 1] == dict_path[i][L - 1]:
            point += 1
    if L - 1 != 0:
        path_add += edge / (L - 1)
    point_add = point / L
    return tor_hits, path_add, point_add


# --------------------------------------------------------------------------- OM step
def om_step(img_raw: torch.Tensor, text_raw: torch.Tensor, log_scale: torch.Tensor,
            c2p, d2n, target: int, *, out_ratio: float, in_ratio: float, weights: str,
            weighting: str, k: int, num_compare: int, layer_weight=None, rng=_random):
    """One OM training step of the head, clip_tree.py:222-281.

    ``img_raw`` [B,D] are un-normalised image features (encoder output), ``text_raw`` [N,D]
    the un-normalised text feature of every node (the reference re-encodes
    ``node_tokens[compare_idx]`` each iteration, :261 -- with a frozen table that is a row
    gather), ``log_scale`` the scalar ``logit_scale`` parameter (logits are multiplied by its
    ``exp``, :263).  Returns a dict with the python-float loss sum (:279), the per-iteration
    losses, the sampled ids, and the gradients the reference leaves on the image features
    clone (:226,:280), the text table and ``logit_scale``.
    """
    img_raw = img_raw.detach().float()
    text = text_raw.detach().float().clone().requires_grad_(True)
    ls = log_scale.detach().float().clone().requires_grad_(True)
    B = img_raw.shape[0]
    img_n = img_raw / img_raw.norm(dim=-1, keepdim=True)          # :225
    img_ = img_n.detach().clone().requires_grad_(True)            # :226
    ce = torch.nn.CrossEntropyLoss()                               # :49
    losses, ids, labels_all, wts = [], [], [], []
    for (k_loop, m_loop, p_out, depth, parents_in, n_out, n_in) in om_schedule(c2p, target, out_ratio, in_ratio):
        compare_idx, labels = get_contra_topk(d2n, p_out, B, depth, parents_in, k, num_compare, rng)
        tf = text[torch.tensor(compare_idx)]
        tf = tf / tf.norm(dim=-1, keepdim=True)                    # :262
        logits = (img_ @ tf.t()) * ls.exp()                        # :263
        if weighting == "out":                                     # :265-273
            w_in = get_weights("equal", n_in)
            w_out = get_weights(weights, n_out, layer_weight)
        elif weighting == "in":
            w_in = get_weights(weights, n_in, layer_weight)
            w_out = get_weights("equal", n_out)
        else:
            w_in = get_weights(weights, n_in, layer_weight)
            w_out = get_weights(weights, n_out, layer_weight)
        wt = w_in[m_loop] * w_out[k_loop]
        loss_j = ce(logits, torch.tensor(labels)) * wt             # :275
        loss_j.backward()                                          # :276
        losses.append(loss_j.item())                               # :277
        ids.append(list(compare_idx))
        labels_all.append(labels[0])
        wts.append(float(wt))
    return {
        "loss": sum(losses),                                       # :279
        "losses": losses,
        "compare_idx": ids,
        "labels": labels_all,
        "weights": wts,
        "d_img_n": img_.grad.clone(),                              # handed to the encoder at :280
        "d_text_raw": text.grad.clone(),
        "d_log_scale": ls.grad.clone(),
    }
