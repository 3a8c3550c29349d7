"""torch-tensor front end of the C ABI (``include/hgr_b200.h``).

PyTorch is plumbing here: it owns device memory and the current stream; every function
below validates tensors, hands raw device pointers to ``libhgr_b200.so`` and returns the
output tensors.  Nothing computes in torch and nothing falls back to the CPU.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _cabi
from ._cabi import (HGR_IMPL_AUTO, HGR_IMPL_SIMT, HGR_IMPL_TCGEN05,  # noqa: F401
                    HGR_IMPL_TCGEN05_EXACT, HGR_IMPL_TCGEN05_NULL, HGR_IMPL_TCGEN05_SKETCH,
                    HGR_HIER_MAX_CHAIN, HGR_MISTAKE_COUNTERS, HGR_NUM_HITS)

_DTYPE_CODE = {torch.float32: _cabi.HGR_F32, torch.bfloat16: _cabi.HGR_BF16, torch.float16: _cabi.HGR_F16}
_workspaces = {}
_retired = []   # outgrown workspaces, kept alive for graphs that captured them


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device (the raw getter is ~20x cheaper than building a
    `torch.cuda.Stream` object -- ten launches per OM step pay for it)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor: hgrnet_b200 has no CPU path" % name)
    if dtype is not None and t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _workspace(nbytes: int, device) -> torch.Tensor:
    key = (device.type, device.index, _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            # a CUDA graph captured on this stream may have baked the old pointer in (EvalStream, ShardedEvalStream;
            # torch hands out pooled stream handles, so another stream object can land on the same key): never free a
            # workspace that has been handed out
            _retired.append(ws)
        ws = torch.zeros(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)   # header words (epoch, counters) start at 0
        _workspaces[key] = ws
    return ws


def last_rescan_count(device=None) -> int:
    """Rows the last tcgen05 ``score_topk`` call on this stream re-scanned exactly (speculative lists that
    could not be certified).  Diagnostics: reads 4 bytes back from the workspace (synchronises)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ws = _workspaces.get((device.type, device.index, _stream()))
    return 0 if ws is None else int(ws[:4].view(torch.int32).item())


def new_hits(device) -> torch.Tensor:
    """Device-resident Hit@{1,2,5,10,20} counters (the reference keeps them on device too, main.py:121,146)."""
    return torch.zeros(HGR_NUM_HITS, dtype=torch.int64, device=device)


def aggregate_normalize(E: torch.Tensor, rowptr: Optional[torch.Tensor] = None,
                        col: Optional[torch.Tensor] = None, w: Optional[torch.Tensor] = None,
                        row_map: Optional[torch.Tensor] = None, out_dtype=torch.bfloat16,
                        return_norm: bool = False):
    """``out[r] = normalize(sum_j w[j] * E[col[j]])`` over CSR row ``row_map[r]`` (identity CSR if ``rowptr is None``).

    model/clip_tree.py:323 / :330 and, with ``row_map = test_index``, the gather of main.py:136.
    """
    lib = _cabi.load()
    E = _require(E, "E")
    if E.dtype not in _DTYPE_CODE:
        raise TypeError("E dtype %s not supported" % E.dtype)
    n_src, D = E.shape
    if rowptr is not None:
        rowptr = _require(rowptr, "rowptr", torch.int32)
        col = _require(col, "col", torch.int32)
        n_rows = rowptr.numel() - 1
        if w is not None:
            w = _require(w, "w", torch.float32)
    else:
        n_rows = n_src
    if row_map is not None:
        row_map = _require(row_map, "row_map", torch.int32)
        n_out = row_map.numel()
    else:
        n_out = n_rows
    out = torch.empty((n_out, D), dtype=out_dtype, device=E.device)
    norm = torch.empty((n_out,), dtype=torch.float32, device=E.device) if return_norm else None
    _cabi.check(lib.hgr_aggregate_normalize(_ptr(E), _DTYPE_CODE[E.dtype], n_src, D, _ptr(rowptr), _ptr(col),
                                            _ptr(w), n_rows, _ptr(row_map), n_out, _ptr(out),
                                            _DTYPE_CODE[out_dtype], _ptr(norm), _stream()))
    return (out, norm) if return_norm else out


def normalize_rows(x: torch.Tensor, out_dtype=torch.bfloat16, return_norm: bool = False):
    """Row L2-normalise (``x / x.norm(dim=-1, keepdim=True)``, model/clip_tree.py:330)."""
    return aggregate_normalize(x, out_dtype=out_dtype, return_norm=return_norm)


def normalize_rows_dual(E: torch.Tensor, out: torch.Tensor, dst_map: Optional[torch.Tensor] = None,
                        out2: Optional[torch.Tensor] = None) -> None:
    """One pass of the bank refresh (clip_tree.py:318-325 + main.py:136): ``out[r] = E[r] / |E[r]|`` (``out``: the
    chunk's rows of the all-node bf16 bank, written in place) and, where ``dst_map[r] >= 0``, the same row into
    ``out2[dst_map[r]]`` (the test-class bank in its own row order)."""
    lib = _cabi.load()
    E = _require(E, "E")
    if E.dtype not in _DTYPE_CODE:
        raise TypeError("E dtype %s not supported" % E.dtype)
    n, D = E.shape
    if out.dtype != torch.bfloat16 or tuple(out.shape) != (n, D) or not out.is_contiguous() or not out.is_cuda:
        raise ValueError("out must be a contiguous CUDA bf16 [n, D] tensor (a row slice of the bank)")
    if (dst_map is None) != (out2 is None):
        raise ValueError("dst_map and out2 go together")
    if dst_map is not None:
        dst_map = _require(dst_map, "dst_map", torch.int32)
        if dst_map.numel() != n or out2.dtype != torch.bfloat16 or out2.shape[1] != D or not out2.is_contiguous():
            raise ValueError("dst_map [n] int32 / out2 bf16 [*, D] contiguous expected")
    _cabi.check(lib.hgr_normalize_rows_dual(_ptr(E), _DTYPE_CODE[E.dtype], n, D, _ptr(out), _ptr(dst_map), _ptr(out2),
                                            _stream()))


def score_topk(X: torch.Tensor, bank: torch.Tensor, *, col_id: Optional[torch.Tensor] = None, id_base: int = 0,
               targets: Optional[torch.Tensor] = None, K: int = 20, scale: float = 1.0,
               hits: Optional[torch.Tensor] = None, impl: int = HGR_IMPL_AUTO,
               out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
               grid_share: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fused logits + per-row sorted top-K (+ Hit@k accumulation into ``hits``).

    model/clip_tree.py:331 + main.py:136-147.  Returns ``(val [B,K] fp32, idx [B,K] int32 node ids)``.
    ``grid_share`` > 1: the call is one of that many batches meant to run at the same time, and the tcgen05 kernel
    takes that share of the CTA pairs (``HGR_IMPL_GRID_SHARE``; same results).
    """
    lib = _cabi.load()
    X = _require(X, "X", torch.bfloat16)
    bank = _require(bank, "bank", torch.bfloat16)
    B, D = X.shape
    C, D2 = bank.shape
    if D != D2:
        raise ValueError("X and bank disagree on D: %d vs %d" % (D, D2))
    if col_id is not None:
        col_id = _require(col_id, "col_id", torch.int32)
        if col_id.numel() != C:
            raise ValueError("col_id must have one entry per bank row")
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
        if targets.numel() != B:
            raise ValueError("targets must have one entry per image row")
    if hits is not None:
        hits = _require(hits, "hits", torch.int64)
    if out is not None:
        val, idx = out
        if val.shape != (B, K) or idx.shape != (B, K) or val.dtype != torch.float32 or idx.dtype != torch.int32 \
                or not val.is_contiguous() or not idx.is_contiguous():
            raise ValueError("out must be contiguous (float32 [B,K], int32 [B,K])")
    else:
        val = torch.empty((B, K), dtype=torch.float32, device=X.device)
        idx = torch.empty((B, K), dtype=torch.int32, device=X.device)
    if not 1 <= grid_share <= _cabi.HGR_GRID_SHARE_MAX:
        raise ValueError("grid_share = %d outside [1, %d]" % (grid_share, _cabi.HGR_GRID_SHARE_MAX))
    if grid_share > 1:
        impl |= grid_share << _cabi.HGR_IMPL_GRID_SHARE_SHIFT
    nbytes = lib.hgr_score_topk_workspace_bytes(B, C, D, K)
    ws = _workspace(nbytes, X.device)
    _cabi.check(lib.hgr_score_topk(_ptr(X), _ptr(bank), _ptr(col_id), id_base, _ptr(targets), B, C, D,
                                   float(scale), K, _ptr(ws), ws.numel(), _ptr(val), _ptr(idx), _ptr(hits),
                                   impl, _stream()))
    return val, idx


def score_topk_splits(X: torch.Tensor, bank: torch.Tensor, group_end, group_splits, n_splits: int, *,
                      col_id: Optional[torch.Tensor] = None, id_base: int = 0, targets: Optional[torch.Tensor] = None,
                      node_splits: Optional[torch.Tensor] = None, counts: Optional[torch.Tensor] = None, K: int = 20,
                      scale: float = 1.0, impl: int = HGR_IMPL_AUTO,
                      out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``score_topk`` for ``n_splits`` test splits in one pass (``hgr_score_topk_splits``, main.py:104-222 once per
    split).  ``bank`` is the union of the splits' classes with the classes of equal membership in contiguous groups:
    ``group_end`` (host ints, exclusive ends, the last = C) and ``group_splits`` (host ints, bit s = the group belongs to
    split s).  ``counts`` (int64 ``[n_splits, HGR_NUM_HITS + 1]``, optional) is incremented by Hit@{1,2,5,10,20} and the
    row count of every split, a row counting toward split s when bit s of ``node_splits[targets[row]]`` (uint8 per node)
    is set.  Returns ``(val [S,B,K] fp32, idx [S,B,K] int32 node ids)``."""
    import ctypes
    lib = _cabi.load()
    X = _require(X, "X", torch.bfloat16)
    bank = _require(bank, "bank", torch.bfloat16)
    B, D = X.shape
    C = bank.shape[0]
    if bank.shape[1] != D:
        raise ValueError("X and bank disagree on D: %d vs %d" % (D, bank.shape[1]))
    n_groups = len(group_end)
    if len(group_splits) != n_groups:
        raise ValueError("group_end and group_splits disagree")
    if col_id is not None:
        col_id = _require(col_id, "col_id", torch.int32)
        if col_id.numel() != C:
            raise ValueError("col_id must have one entry per bank row")
    if counts is not None:
        if targets is None or node_splits is None:
            raise ValueError("counts need targets and node_splits")
        if not counts.is_cuda or counts.dtype != torch.int64 or counts.numel() != n_splits * (HGR_NUM_HITS + 1) \
                or not counts.is_contiguous():
            raise ValueError("counts must be a contiguous CUDA int64 [%d, %d] tensor" % (n_splits, HGR_NUM_HITS + 1))
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
        if targets.numel() != B:
            raise ValueError("targets must have one entry per image row")
    if node_splits is not None:
        node_splits = _require(node_splits, "node_splits", torch.uint8)
    if out is not None:
        val, idx = out
        if val.shape != (n_splits, B, K) or idx.shape != (n_splits, B, K) or val.dtype != torch.float32 \
                or idx.dtype != torch.int32 or not val.is_contiguous() or not idx.is_contiguous():
            raise ValueError("out must be contiguous (float32 [S,B,K], int32 [S,B,K])")
    else:
        val = torch.empty((n_splits, B, K), dtype=torch.float32, device=X.device)
        idx = torch.empty((n_splits, B, K), dtype=torch.int32, device=X.device)
    ends = (ctypes.c_int32 * n_groups)(*[int(e) for e in group_end])
    gsp = (ctypes.c_uint8 * n_groups)(*[int(m) for m in group_splits])
    nbytes = lib.hgr_score_topk_splits_workspace_bytes(B, C, D, K, n_groups, ends)
    ws = _workspace(nbytes, X.device)      # the stream's scoring workspace: last_rescan_count() reads it
    n_nodes = node_splits.numel() if node_splits is not None else 0
    _cabi.check(lib.hgr_score_topk_splits(_ptr(X), _ptr(bank), _ptr(col_id), id_base, _ptr(targets), _ptr(node_splits),
                                          n_nodes, B, C, D, float(scale), K, n_groups, ends, gsp, n_splits, _ptr(ws),
                                          ws.numel(), _ptr(val), _ptr(idx), _ptr(counts), impl, _stream()))
    return val, idx


def score_topk_plan(B: int, C: int, D: int, K: int = 20, grid_share: int = 1) -> dict:
    """What ``score_topk`` would do for this shape on the tcgen05 path at ``grid_share`` (no launch, works without a
    GPU)."""
    import ctypes
    plan = (ctypes.c_int32 * 8)()
    _cabi.check(_cabi.load().hgr_score_topk_plan_shared(B, C, D, K, grid_share, plan))
    keys = ("workers", "row_tiles", "units_per_row_tile", "lists_per_row", "list_len", "warps_per_quarter",
            "ring_depth", "cols_per_worker")
    return dict(zip(keys, list(plan)))


def score_topk_grid_share(B: int, C: int, D: int, K: int = 20) -> int:
    """The ``grid_share`` the library recommends for a batch of this shape that runs beside others (host only)."""
    return int(_cabi.load().hgr_score_topk_grid_share(B, C, D, K))


def score_topk_footprint(B: int, C: int, D: int, K: int = 20, x_dtype=torch.bfloat16, grid_share: int = 1) -> dict:
    """What one batch of ``normalize_rows`` + ``score_topk`` (at ``grid_share``) asks of an SM, per kernel
    (``normalize``, ``score``, ``merge``): ``{threads, registers, static_smem, dynamic_smem}`` (registers per thread,
    bytes).  Needs a device."""
    import ctypes
    out = (ctypes.c_int32 * 12)()
    _cabi.check(_cabi.load().hgr_score_topk_footprint_shared(B, C, D, K, grid_share, _DTYPE_CODE[x_dtype], out))
    keys = ("threads", "registers", "static_smem", "dynamic_smem")
    return {name: dict(zip(keys, list(out)[4 * i:4 * i + 4])) for i, name in enumerate(("normalize", "score", "merge"))}


def topk_merge(part_val: torch.Tensor, part_idx: torch.Tensor, *, targets: Optional[torch.Tensor] = None,
               hits: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge ``[P, B, K]`` partial lists (node ids) into the final ``[B, K]`` top-K + hits.

    The two inputs may be strided views of one gathered buffer (same part stride, dense ``[B, K]`` inside).
    """
    lib = _cabi.load()
    if part_val.dtype != torch.float32 or part_idx.dtype != torch.int32 or not part_val.is_cuda:
        raise TypeError("part_val/part_idx must be CUDA float32/int32 tensors")
    P, B, K = part_val.shape
    dense_inner = lambda t: t.stride(2) == 1 and t.stride(1) == K
    if not (dense_inner(part_val) and dense_inner(part_idx) and part_val.stride(0) == part_idx.stride(0)):
        part_val, part_idx = part_val.contiguous(), part_idx.contiguous()
    part_stride = part_val.stride(0) if P > 1 else 0
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
    if hits is not None:
        hits = _require(hits, "hits", torch.int64)
    val = torch.empty((B, K), dtype=torch.float32, device=part_val.device)
    idx = torch.empty((B, K), dtype=torch.int32, device=part_val.device)
    _cabi.check(lib.hgr_topk_merge(_ptr(part_val), _ptr(part_idx), P, B, K, part_stride, _ptr(targets), _ptr(val),
                                   _ptr(idx), _ptr(hits), _stream()))
    return val, idx


def topk_merge_raw(part_val_ptr: int, part_idx_ptr: int, P: int, B: int, K: int, part_stride: int, device, *,
                   targets: Optional[torch.Tensor] = None, hits: Optional[torch.Tensor] = None,
                   out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``topk_merge`` on raw device pointers (lists that live in a peer-exchange buffer, see ``dist.PeerExchange``)."""
    lib = _cabi.load()
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
    if hits is not None:
        hits = _require(hits, "hits", torch.int64)
    if out is None:
        out = (torch.empty((B, K), dtype=torch.float32, device=device), torch.empty((B, K), dtype=torch.int32, device=device))
    _cabi.check(lib.hgr_topk_merge(part_val_ptr, part_idx_ptr, P, B, K, part_stride, _ptr(targets), _ptr(out[0]),
                                   _ptr(out[1]), _ptr(hits), _stream()))
    return out


def score_topk_scatter(X: torch.Tensor, bank: torch.Tensor, val_block_ptrs, idx_block_ptrs, block_rows: int, *,
                       col_id: Optional[torch.Tensor] = None, id_base: int = 0, K: int = 20, scale: float = 1.0,
                       impl: int = HGR_IMPL_AUTO, bound_block_ptrs=None, C_total: int = 0) -> None:
    """``score_topk`` whose final lists of rows ``[g*block_rows, (g+1)*block_rows)`` are written to the dense
    ``[block_rows, K]`` arrays at ``val_block_ptrs[g]`` / ``idx_block_ptrs[g]`` (device pointers, local or peer).

    With ``bound_block_ptrs`` (``[block_rows]`` fp32 arrays) and ``C_total`` the bank is one shard of a row's global
    stream of ``C_total`` classes: narrow lists sized for the GLOBAL certificate, no local repair, and per row an upper
    bound of everything the shard dropped (``hgr_score_topk_scatter_bounded``; the owner runs
    ``topk_merge_certified``)."""
    import ctypes
    lib = _cabi.load()
    X = _require(X, "X", torch.bfloat16)
    bank = _require(bank, "bank", torch.bfloat16)
    B, D = X.shape
    C = bank.shape[0]
    if col_id is not None:
        col_id = _require(col_id, "col_id", torch.int32)
    n = len(val_block_ptrs)
    if len(idx_block_ptrs) != n:
        raise ValueError("val/idx block tables disagree")
    vt = (ctypes.c_void_p * n)(*val_block_ptrs)
    it = (ctypes.c_void_p * n)(*idx_block_ptrs)
    nbytes = lib.hgr_score_topk_workspace_bytes(B, C, D, K)
    ws = _workspace(nbytes, X.device)
    if bound_block_ptrs is not None:
        if len(bound_block_ptrs) != n:
            raise ValueError("bound block table disagrees with the val/idx tables")
        bt = (ctypes.c_void_p * n)(*bound_block_ptrs)
        _cabi.check(lib.hgr_score_topk_scatter_bounded(_ptr(X), _ptr(bank), _ptr(col_id), id_base, B, C, D, float(scale),
                                                       K, _ptr(ws), ws.numel(), block_rows, n, vt, it, bt,
                                                       int(C_total), impl, _stream()))
        return
    _cabi.check(lib.hgr_score_topk_scatter(_ptr(X), _ptr(bank), _ptr(col_id), id_base, B, C, D, float(scale), K,
                                           _ptr(ws), ws.numel(), block_rows, n, vt, it, impl, _stream()))


def global_list_len(B: int, C: int, D: int, K: int, C_total: int) -> int:
    """Entries per list ``score_topk_scatter`` keeps for a shard of ``C`` of ``C_total`` classes (host only)."""
    r = _cabi.load().hgr_score_topk_global_list_len(B, C, D, K, C_total)
    if r < 0:
        _cabi.check(r)
    return int(r)


def _split_tables(group_end, group_splits, split_C_total):
    import ctypes
    n_groups, S = len(group_end), len(split_C_total)
    if len(group_splits) != n_groups:
        raise ValueError("group_end and group_splits disagree")
    return ((ctypes.c_int32 * max(n_groups, 1))(*[int(e) for e in group_end]),
            (ctypes.c_uint8 * max(n_groups, 1))(*[int(m) for m in group_splits]),
            (ctypes.c_int64 * S)(*[int(c) for c in split_C_total]))


def score_topk_splits_scatter(X: torch.Tensor, bank: torch.Tensor, group_end, group_splits, split_C_total,
                              val_block_ptrs, idx_block_ptrs, bound_block_ptrs, block_rows: int, split_stride: int, *,
                              col_id: Optional[torch.Tensor] = None, id_base: int = 0, K: int = 20,
                              scale: float = 1.0) -> None:
    """Producer of the class-sharded multi-split head (``hgr_score_topk_splits_scatter_bounded``, main.py:104-222 once
    per split): ``bank`` is this rank's part of the union bank with its own group table (``group_end`` / ``group_splits``,
    host ints, as ``score_topk_splits``; empty for a rank without rows), ``split_C_total`` the GLOBAL class count of every
    split.  Per split s the rank's top-K of rows ``[g*block_rows, (g+1)*block_rows)`` and the bound of what it dropped go
    to ``val_block_ptrs[g]`` / ``idx_block_ptrs[g]`` / ``bound_block_ptrs[g]`` + ``s * split_stride`` elements (device
    pointers, local or peer); the owner runs ``topk_merge_splits_certified``."""
    lib = _cabi.load()
    X = _require(X, "X", torch.bfloat16)
    B, D = X.shape
    C = bank.shape[0]
    if C:
        bank = _require(bank, "bank", torch.bfloat16)
        if bank.shape[1] != D:
            raise ValueError("X and bank disagree on D: %d vs %d" % (D, bank.shape[1]))
    if col_id is not None:
        col_id = _require(col_id, "col_id", torch.int32)
        if col_id.numel() != C:
            raise ValueError("col_id must have one entry per bank row")
    n = len(val_block_ptrs)
    if len(idx_block_ptrs) != n or len(bound_block_ptrs) != n:
        raise ValueError("val/idx/bound block tables disagree")
    import ctypes
    vt = (ctypes.c_void_p * n)(*val_block_ptrs)
    it = (ctypes.c_void_p * n)(*idx_block_ptrs)
    bt = (ctypes.c_void_p * n)(*bound_block_ptrs)
    ends, gsp, ctot = _split_tables(group_end, group_splits, split_C_total)
    n_groups = len(group_end)
    nbytes = lib.hgr_score_topk_splits_scatter_bounded_workspace_bytes(B, C, D, K, n_groups, ends)
    ws = _workspace(nbytes, X.device)
    _cabi.check(lib.hgr_score_topk_splits_scatter_bounded(_ptr(X), _ptr(bank) if C else None, _ptr(col_id), id_base, B, C,
                                                          D, float(scale), K, n_groups, ends, gsp, len(split_C_total),
                                                          ctot, _ptr(ws), ws.numel(), block_rows, n, vt, it, bt,
                                                          int(split_stride), HGR_IMPL_AUTO, _stream()))


def splits_global_list_len(B: int, C: int, D: int, K: int, group_end, group_splits, split_C_total) -> int:
    """Entries per list ``score_topk_splits_scatter`` keeps on a rank's part of the union bank (host only)."""
    ends, gsp, ctot = _split_tables(group_end, group_splits, split_C_total)
    r = _cabi.load().hgr_score_topk_splits_global_list_len(B, C, D, K, len(group_end), ends, gsp, len(split_C_total), ctot)
    if r < 0:
        _cabi.check(r)
    return int(r)


def topk_merge_splits_certified(part_val_ptr: int, part_idx_ptr: int, part_bound_ptr: int, P: int, B: int, K: int,
                                n_splits: int, part_stride: int, bound_stride: int, split_stride: int,
                                x_rows: torch.Tensor, shards: torch.Tensor, node_splits: torch.Tensor, device, *,
                                scale: float = 1.0, targets: Optional[torch.Tensor] = None,
                                counts: Optional[torch.Tensor] = None, repair_count: Optional[torch.Tensor] = None,
                                out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Owner side of the class-sharded multi-split head (``hgr_topk_merge_splits_certified``): per split, merge the
    ``P`` shard lists of ``B`` rows, certify against the shards' bounds and repair the rest exactly from ``shards``
    (``shard_table``) with the rows' features ``x_rows [B, D]`` bf16.  ``counts`` int64 ``[n_splits, HGR_NUM_HITS + 1]``
    as in ``score_topk_splits``.  Returns ``(val [S,B,K], idx [S,B,K])``."""
    lib = _cabi.load()
    x_rows = _require(x_rows, "x_rows", torch.bfloat16)
    if x_rows.shape[0] != B:
        raise ValueError("x_rows must hold the %d rows being merged" % B)
    if shards.dtype != torch.int64 or tuple(shards.shape) != (P, 4) or not shards.is_cuda:
        raise ValueError("shards must be the [P, 4] int64 device tensor shard_table() builds")
    node_splits = _require(node_splits, "node_splits", torch.uint8)
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
    if counts is not None and (not counts.is_cuda or counts.dtype != torch.int64 or not counts.is_contiguous()
                               or counts.numel() != n_splits * (HGR_NUM_HITS + 1)):
        raise ValueError("counts must be a contiguous CUDA int64 [%d, %d] tensor" % (n_splits, HGR_NUM_HITS + 1))
    if repair_count is not None:
        repair_count = _require(repair_count, "repair_count", torch.int32)
    if out is None:
        out = (torch.empty((n_splits, B, K), dtype=torch.float32, device=device),
               torch.empty((n_splits, B, K), dtype=torch.int32, device=device))
    _cabi.check(lib.hgr_topk_merge_splits_certified(part_val_ptr, part_idx_ptr, part_bound_ptr, P, B, K, n_splits,
                                                    part_stride, bound_stride, split_stride, _ptr(targets),
                                                    _ptr(node_splits), node_splits.numel(), _ptr(out[0]), _ptr(out[1]),
                                                    _ptr(counts), _ptr(x_rows), x_rows.shape[1], _ptr(shards),
                                                    float(scale), _ptr(repair_count), _stream()))
    return out


def shard_table(shards, device) -> torch.Tensor:
    """Device copy of an ``hgr_shard_t`` array: ``shards`` = [(bank pointer, col_id pointer or 0, C, id_base), ...]
    (32 bytes per entry: two pointers, int64 C, int32 id_base + padding)."""
    rows = [[int(b), int(c or 0), int(n), int(base) & 0xFFFFFFFF] for (b, c, n, base) in shards]
    return torch.tensor(rows, dtype=torch.int64).to(device)


def topk_merge_certified(part_val_ptr: int, part_idx_ptr: int, part_bound_ptr: int, P: int, B: int, K: int,
                         part_stride: int, bound_stride: int, x_rows: torch.Tensor, shards: torch.Tensor, device, *,
                         scale: float = 1.0, targets: Optional[torch.Tensor] = None,
                         hits: Optional[torch.Tensor] = None, repair_count: Optional[torch.Tensor] = None,
                         out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Owner side of the global certificate (``hgr_topk_merge_certified``): merge the ``P`` shard lists of ``B`` rows,
    certify every row against the shards' bounds, repair the rest exactly from ``shards`` (``shard_table``) with the
    rows' normalised features ``x_rows [B, D]`` bf16."""
    lib = _cabi.load()
    x_rows = _require(x_rows, "x_rows", torch.bfloat16)
    if x_rows.shape[0] != B:
        raise ValueError("x_rows must hold the %d rows being merged" % B)
    if shards.dtype != torch.int64 or tuple(shards.shape) != (P, 4) or not shards.is_cuda:
        raise ValueError("shards must be the [P, 4] int64 device tensor shard_table() builds")
    if targets is not None:
        targets = _require(targets, "targets", torch.int32)
    if hits is not None:
        hits = _require(hits, "hits", torch.int64)
    if repair_count is not None:
        repair_count = _require(repair_count, "repair_count", torch.int32)
    if out is None:
        out = (torch.empty((B, K), dtype=torch.float32, device=device), torch.empty((B, K), dtype=torch.int32, device=device))
    _cabi.check(lib.hgr_topk_merge_certified(part_val_ptr, part_idx_ptr, part_bound_ptr, P, B, K, part_stride, bound_stride,
                                             _ptr(targets), _ptr(out[0]), _ptr(out[1]), _ptr(hits), _ptr(x_rows),
                                             x_rows.shape[1], _ptr(shards), float(scale), _ptr(repair_count), _stream()))
    return out


def peer_alloc(nbytes: int) -> Tuple[int, bytes]:
    """cudaMalloc'd, zeroed exchange buffer on the current device + its CUDA IPC handle."""
    import ctypes
    lib = _cabi.load()
    ptr = ctypes.c_void_p()
    handle = (ctypes.c_ubyte * 64)()
    _cabi.check(lib.hgr_peer_alloc(nbytes, ctypes.byref(ptr), handle))
    return int(ptr.value), bytes(handle)


def peer_open(handle: bytes) -> int:
    import ctypes
    lib = _cabi.load()
    ptr = ctypes.c_void_p()
    buf = (ctypes.c_ubyte * 64)(*handle)
    _cabi.check(lib.hgr_peer_open(buf, ctypes.byref(ptr)))
    return int(ptr.value)


def peer_close(ptr: int) -> None:
    _cabi.check(_cabi.load().hgr_peer_close(ptr))


def peer_free(ptr: int) -> None:
    _cabi.check(_cabi.load().hgr_peer_free(ptr))


def normalize_rows_bcast(x_block: torch.Tensor, row0: int, dst_ptrs) -> None:
    """Normalise the rows of ``x_block`` and store row r at row ``row0 + r`` of every bf16 ``[*, D]`` array in
    ``dst_ptrs`` (device pointers, local or peer)."""
    import ctypes
    x_block = _require(x_block, "x_block")
    if x_block.dtype not in _DTYPE_CODE:
        raise TypeError("x_block dtype %s not supported" % x_block.dtype)
    n, D = x_block.shape
    dt = (ctypes.c_void_p * len(dst_ptrs))(*dst_ptrs)
    _cabi.check(_cabi.load().hgr_normalize_rows_bcast(_ptr(x_block), _DTYPE_CODE[x_block.dtype], n, D, row0,
                                                      len(dst_ptrs), dt, _stream()))


def peer_signal(flag_ptrs, seq: torch.Tensor) -> None:
    """Publish this rank's next sequence number (``seq`` is a 1-element int32 device counter) to ``flag_ptrs``."""
    import ctypes
    n = len(flag_ptrs)
    ft = (ctypes.c_void_p * n)(*flag_ptrs)
    _cabi.check(_cabi.load().hgr_peer_signal(ft, n, _ptr(seq), _stream()))


def peer_wait(flags_ptr: int, n: int, seq: torch.Tensor) -> None:
    """Advance the consumer counter ``seq`` and wait until the ``n`` local flag words have reached it."""
    _cabi.check(_cabi.load().hgr_peer_wait(flags_ptr, n, _ptr(seq), _stream()))


def logits_dense(X: torch.Tensor, bank: torch.Tensor, scale: float = 1.0, impl: int = HGR_IMPL_AUTO,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``scale * X @ bank.T`` in fp32 (model/clip_tree.py:331 / :263) on the tcgen05 main loop.
    ``out`` (optional): fp32 ``[B, C]`` on X's device with unit column stride and, when B > 1, stride(0) >= C; its rows
    may be further apart than C (a column slice of a wider buffer), the cells between them are left untouched."""
    lib = _cabi.load()
    X = _require(X, "X", torch.bfloat16)
    bank = _require(bank, "bank", torch.bfloat16)
    B, D = X.shape
    C = bank.shape[0]
    if out is None:
        out = torch.empty((B, C), dtype=torch.float32, device=X.device)
    elif out.dtype != torch.float32 or out.device != X.device or tuple(out.shape) != (B, C) or out.stride(1) != 1 \
            or (B > 1 and out.stride(0) < C):
        raise ValueError("out must be a float32 [%d, %d] tensor on %s with stride(1) == 1 and stride(0) >= %d, got %s %s "
                         "on %s with strides %s" % (B, C, X.device, C, out.dtype, list(out.shape), out.device,
                                                     list(out.stride())))
    ldo = out.stride(0) if B > 1 else C        # one row: its stride is never used
    _cabi.check(lib.hgr_logits_dense(_ptr(X), _ptr(bank), B, C, D, float(scale), _ptr(out), ldo, impl, _stream()))
    return out


def _hier_workspace(nbytes: int, device) -> torch.Tensor:
    """Per-stream scratch of the fused TOR / POR calls: zero when allocated, handed back zeroed by every call (the
    scoring kernel's workspace on the same stream keeps header words, so this is a separate buffer)."""
    key = ("hier", device.index, _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            _retired.append(ws)
        ws = torch.zeros(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def new_hier_counts(device, n_sets: Optional[int] = None) -> torch.Tensor:
    """Zeroed per-chain-length counters of ``hier_metrics_fused_rows``: int64 ``[HGR_HIER_MAX_CHAIN + 1, 4]``, or
    ``[n_sets, HGR_HIER_MAX_CHAIN + 1, 4]`` with ``n_sets``; bin L = ``{rows, TOR hits, points, edges}`` of the rows whose
    label chain has L entries."""
    shape = (HGR_HIER_MAX_CHAIN + 1, 4)
    return torch.zeros(shape if n_sets is None else (n_sets, *shape), dtype=torch.int64, device=device)


def _hier_sets(counts: torch.Tensor, node_splits: Optional[torch.Tensor], n_nodes: int):
    """The counter sets of a TOR / POR call: ``counts`` ``[33, 4]`` or ``[S, 33, 4]`` (``new_hier_counts``), S > 1 only
    with ``node_splits`` (uint8 per node).  Returns ``(S, node_splits)``."""
    if not counts.is_cuda:
        raise ValueError("counts must be a CUDA tensor: hgrnet_b200 has no CPU path")
    if counts.dtype != torch.int64 or counts.dim() not in (2, 3) or tuple(counts.shape[-2:]) != (HGR_HIER_MAX_CHAIN + 1, 4) \
            or not counts.is_contiguous():
        raise ValueError("counts must be a contiguous int64 [%d, 4] or [S, %d, 4] tensor (new_hier_counts)"
                         % (HGR_HIER_MAX_CHAIN + 1, HGR_HIER_MAX_CHAIN + 1))
    S = counts.shape[0] if counts.dim() == 3 else 1
    if node_splits is not None:
        node_splits = _require(node_splits, "node_splits", torch.uint8)
        if node_splits.numel() != n_nodes:
            raise ValueError("node_splits must have one entry per node")
    elif S != 1:
        raise ValueError("%d counter sets need node_splits" % S)
    return S, node_splits


def _check_rows_out(lvl_idx, top1, B: int, n_levels: int) -> None:
    for name, t, shape in (("lvl_idx", lvl_idx, (B, n_levels)), ("top1", top1, (B,))):
        if t is not None and (t.dtype != torch.int32 or tuple(t.shape) != shape or not t.is_contiguous() or not t.is_cuda):
            raise ValueError("%s must be a contiguous CUDA int32 %s tensor" % (name, list(shape)))


def hier_metrics_fused_rows(x_norm: torch.Tensor, bank_sorted: torch.Tensor, level_end, sorted_to_pos: torch.Tensor,
                            first_out: torch.Tensor, targets: torch.Tensor, chain_ptr: torch.Tensor,
                            chain_pos: torch.Tensor, chain_level: torch.Tensor, counts: torch.Tensor,
                            node_splits: Optional[torch.Tensor] = None, lvl_idx: Optional[torch.Tensor] = None,
                            top1: Optional[torch.Tensor] = None) -> None:
    """TOR / POR counters (main.py:143,152-191) of one batch without the dense logits: ``bank_sorted`` holds the train
    rows of the bank sorted by level (``level_end``: host list of exclusive ends), the per-level arg-max runs in the
    epilogue of the tcgen05 GEMM.  Row i is matched against the chain of node ``targets[i]``, read from the chain table
    ``chain_ptr [n_nodes + 1]`` / ``chain_pos`` / ``chain_level`` (``evaluate.chain_table``).  Positions (chain_pos,
    first_out, lvl_idx, top1) are positions in ``train_index``.  ``counts`` (``new_hier_counts``) is incremented per
    chain length; rows whose target is outside ``[0, n_nodes)`` are counted nowhere.  With ``node_splits`` (uint8 per
    node) ``counts`` may be ``[S, 33, 4]``: a row is added to set s for every bit s of ``node_splits[targets[row]]``,
    from one GEMM whatever S is.  No host work depends on the batch's contents, so the call can be captured in a CUDA
    graph.  See ``hgr_hier_metrics_fused_rows`` in the header."""
    import ctypes
    lib = _cabi.load()
    x_norm = _require(x_norm, "x_norm", torch.bfloat16)
    bank_sorted = _require(bank_sorted, "bank_sorted", torch.bfloat16)
    sorted_to_pos = _require(sorted_to_pos, "sorted_to_pos", torch.int32)
    first_out = _require(first_out, "first_out", torch.int32)
    targets = _require(targets, "targets", torch.int32)
    chain_ptr = _require(chain_ptr, "chain_ptr", torch.int32)
    chain_pos = _require(chain_pos, "chain_pos", torch.int32)
    chain_level = _require(chain_level, "chain_level", torch.int32)
    n_nodes = chain_ptr.numel() - 1
    S, node_splits = _hier_sets(counts, node_splits, n_nodes)
    B, D = x_norm.shape
    M = bank_sorted.shape[0]
    n_levels = len(level_end)
    if sorted_to_pos.numel() != M or first_out.numel() != n_levels or targets.numel() != B \
            or chain_pos.numel() != chain_level.numel():
        raise ValueError("hier_metrics_fused_rows: inconsistent sizes")
    _check_rows_out(lvl_idx, top1, B, n_levels)
    ends = (ctypes.c_int32 * n_levels)(*[int(e) for e in level_end])
    ws = _hier_workspace(B * n_levels * 8, x_norm.device)
    _cabi.check(lib.hgr_hier_metrics_fused_rows(_ptr(x_norm), _ptr(bank_sorted), B, M, D, ends, n_levels,
                                                _ptr(sorted_to_pos), _ptr(first_out), _ptr(targets), n_nodes,
                                                _ptr(chain_ptr), _ptr(chain_pos), _ptr(chain_level), _ptr(node_splits),
                                                S, _ptr(ws), ws.numel(), _ptr(lvl_idx), _ptr(top1), _ptr(counts),
                                                _stream()))


def hier_level_scatter(x_norm: torch.Tensor, bank_shard: torch.Tensor, level_end_local, row_base: int, dst_block_ptrs,
                       block_rows: int) -> None:
    """Producer half of class-sharded TOR / POR (``hgr_hier_level_scatter``): the per-level arg-max of ``x_norm``
    against ``bank_shard`` (sorted rows ``[row_base, row_base + M_r)`` of the level-sorted train bank, ``level_end_local``
    the global level ends clipped to it), each winner word rebased to the global sorted row and stored at the owner of
    its row: rows ``[g*block_rows, (g+1)*block_rows)`` go to the ``[block_rows, n_levels]`` uint64 array at
    ``dst_block_ptrs[g]`` (device pointers, local or peer).  An empty shard stores zeros."""
    import ctypes
    lib = _cabi.load()
    x_norm = _require(x_norm, "x_norm", torch.bfloat16)
    bank_shard = _require(bank_shard, "bank_shard", torch.bfloat16)
    B, D = x_norm.shape
    M_r = bank_shard.shape[0]
    if M_r and bank_shard.shape[1] != D:
        raise ValueError("x_norm and bank_shard disagree on D: %d vs %d" % (D, bank_shard.shape[1]))
    n_levels = len(level_end_local)
    ends = (ctypes.c_int32 * n_levels)(*[int(e) for e in level_end_local])
    n = len(dst_block_ptrs)
    dt = (ctypes.c_void_p * n)(*dst_block_ptrs)
    ws = _hier_workspace(B * n_levels * 8, x_norm.device)
    _cabi.check(lib.hgr_hier_level_scatter(_ptr(x_norm), _ptr(bank_shard), B, M_r, D, ends, n_levels, int(row_base),
                                           _ptr(ws), ws.numel(), block_rows, n, dt, _stream()))


def hier_finish_rows_gathered(parts_ptr: int, n_parts: int, part_stride: int, n_rows: int, M: int, n_levels: int,
                              sorted_to_pos: torch.Tensor, first_out: torch.Tensor, targets: torch.Tensor,
                              chain_ptr: torch.Tensor, chain_pos: torch.Tensor, chain_level: torch.Tensor,
                              counts: torch.Tensor, node_splits: Optional[torch.Tensor] = None,
                              lvl_idx: Optional[torch.Tensor] = None, top1: Optional[torch.Tensor] = None) -> None:
    """Owner half of class-sharded TOR / POR (``hgr_hier_finish_rows_gathered``): for ``n_rows`` rows, the max over the
    ``n_parts`` shards' winner words at ``parts_ptr`` (``part_stride`` words apart, e.g. a peer-exchange slot), then
    what ``hier_metrics_fused_rows`` does with its own words.  ``targets`` / ``lvl_idx`` / ``top1`` cover these rows;
    ``M``, ``sorted_to_pos``, ``first_out`` and the chain table are the global ones; ``counts`` / ``node_splits`` as in
    ``hier_metrics_fused_rows``."""
    lib = _cabi.load()
    sorted_to_pos = _require(sorted_to_pos, "sorted_to_pos", torch.int32)
    first_out = _require(first_out, "first_out", torch.int32)
    targets = _require(targets, "targets", torch.int32)
    chain_ptr = _require(chain_ptr, "chain_ptr", torch.int32)
    chain_pos = _require(chain_pos, "chain_pos", torch.int32)
    chain_level = _require(chain_level, "chain_level", torch.int32)
    n_nodes = chain_ptr.numel() - 1
    S, node_splits = _hier_sets(counts, node_splits, n_nodes)
    if sorted_to_pos.numel() != M or first_out.numel() != n_levels or targets.numel() != n_rows \
            or chain_pos.numel() != chain_level.numel():
        raise ValueError("hier_finish_rows_gathered: inconsistent sizes")
    _check_rows_out(lvl_idx, top1, n_rows, n_levels)
    _cabi.check(lib.hgr_hier_finish_rows_gathered(parts_ptr, n_parts, part_stride, n_rows, M, n_levels, _ptr(sorted_to_pos),
                                                  _ptr(first_out), _ptr(targets), n_nodes, _ptr(chain_ptr),
                                                  _ptr(chain_pos), _ptr(chain_level), _ptr(node_splits), S,
                                                  _ptr(lvl_idx), _ptr(top1), _ptr(counts), _stream()))


def new_mistake_counts(device, n_sets: int = 1) -> torch.Tensor:
    """Zeroed counters of ``hier_mistakes``: int64 ``[n_sets, HGR_MISTAKE_COUNTERS]`` (rows, mistakes, sums of h and of d
    over the first 1/2/5/10/20 entries, histogram of d at top-1; see ``hgr_hier_mistakes`` in the header)."""
    return torch.zeros((n_sets, HGR_MISTAKE_COUNTERS), dtype=torch.int64, device=device)


def hier_mistakes(idx: torch.Tensor, targets: torch.Tensor, chain_ptr: torch.Tensor, chain_node: torch.Tensor,
                  counts: torch.Tensor, node_splits: Optional[torch.Tensor] = None) -> None:
    """Mistake severity and LCA distance@k counters (``hgr_hier_mistakes``) of top-K lists on the device: ``idx`` int32
    node ids ``[B, K]`` (one set) or ``[S, B, K]`` (one set per test split, with ``node_splits``: list set s counts a row
    only when bit s of ``node_splits[targets[row]]`` is set).  ``targets`` [B] node ids, row by row; ``chain_ptr`` /
    ``chain_node`` the chain table of ``evaluate.chain_csr``.  ``counts`` (``new_mistake_counts(device, S)``) is
    incremented.  No host work depends on the batch: the call can be captured in a CUDA graph."""
    lib = _cabi.load()
    if idx.dim() == 2:
        idx = idx.unsqueeze(0)
    if idx.dim() != 3 or idx.dtype != torch.int32 or not idx.is_cuda:
        raise ValueError("idx must be a CUDA int32 [B, K] or [S, B, K] tensor")
    if not (idx.stride(2) == 1 and idx.stride(1) == idx.shape[2]):
        idx = idx.contiguous()
    S, B, K = idx.shape
    targets = _require(targets, "targets", torch.int32)
    chain_ptr = _require(chain_ptr, "chain_ptr", torch.int32)
    chain_node = _require(chain_node, "chain_node", torch.int32)
    if node_splits is not None:
        node_splits = _require(node_splits, "node_splits", torch.uint8)
        if node_splits.numel() != chain_ptr.numel() - 1:
            raise ValueError("node_splits must have one entry per node")
    elif S != 1:
        raise ValueError("%d list sets need node_splits" % S)
    if targets.numel() != B:
        raise ValueError("targets must have one entry per list row")
    if not counts.is_cuda or counts.dtype != torch.int64 or counts.numel() != S * HGR_MISTAKE_COUNTERS \
            or not counts.is_contiguous():
        raise ValueError("counts must be a contiguous CUDA int64 [%d, %d] tensor (new_mistake_counts)"
                         % (S, HGR_MISTAKE_COUNTERS))
    _cabi.check(lib.hgr_hier_mistakes(_ptr(idx), B, K, idx.stride(0) if S > 1 else B * K, S, _ptr(targets),
                                      _ptr(node_splits), _ptr(chain_ptr), _ptr(chain_node), chain_ptr.numel() - 1,
                                      _ptr(counts), _stream()))


def new_class_counts(device, n_nodes: int, n_sets: int = 1) -> torch.Tensor:
    """Zeroed counters of ``class_hits``: int64 ``[n_sets, n_nodes, HGR_NUM_HITS + 1]``, per class
    ``[Hit@1, Hit@2, Hit@5, Hit@10, Hit@20, rows]`` (see ``hgr_class_hits`` in the header)."""
    return torch.zeros((n_sets, n_nodes, HGR_NUM_HITS + 1), dtype=torch.int64, device=device)


def class_hits(idx: torch.Tensor, targets: torch.Tensor, counts: torch.Tensor,
               node_splits: Optional[torch.Tensor] = None) -> None:
    """Per-class Hit@{1,2,5,10,20} and row counters (``hgr_class_hits``) of top-K lists on the device: ``idx`` int32
    node ids ``[B, K]`` (one set) or ``[S, B, K]`` (one set per test split, with ``node_splits``: list set s counts a
    row only when bit s of ``node_splits[targets[row]]`` is set).  ``targets`` [B] node ids, row by row; a row whose
    label is outside ``[0, n_nodes)`` counts nowhere.  ``counts`` (``new_class_counts(device, n_nodes, S)``) is
    incremented.  No host work depends on the batch: the call can be captured in a CUDA graph."""
    lib = _cabi.load()
    if idx.dim() == 2:
        idx = idx.unsqueeze(0)
    if idx.dim() != 3 or idx.dtype != torch.int32 or not idx.is_cuda:
        raise ValueError("idx must be a CUDA int32 [B, K] or [S, B, K] tensor")
    if not (idx.stride(2) == 1 and idx.stride(1) == idx.shape[2]):
        idx = idx.contiguous()
    S, B, K = idx.shape
    targets = _require(targets, "targets", torch.int32)
    if not counts.is_cuda or counts.dtype != torch.int64 or counts.dim() != 3 or counts.shape[0] != S \
            or counts.shape[2] != HGR_NUM_HITS + 1 or not counts.is_contiguous():
        raise ValueError("counts must be a contiguous CUDA int64 [%d, n_nodes, %d] tensor (new_class_counts)"
                         % (S, HGR_NUM_HITS + 1))
    n_nodes = counts.shape[1]
    if node_splits is not None:
        node_splits = _require(node_splits, "node_splits", torch.uint8)
        if node_splits.numel() != n_nodes:
            raise ValueError("node_splits must have one entry per node")
    elif S != 1:
        raise ValueError("%d list sets need node_splits" % S)
    if targets.numel() != B:
        raise ValueError("targets must have one entry per list row")
    _cabi.check(lib.hgr_class_hits(_ptr(idx), B, K, idx.stride(0) if S > 1 else B * K, S, _ptr(targets),
                                   _ptr(node_splits), n_nodes, _ptr(counts), _stream()))


def masked_ce(logits: torch.Tensor, set_ptr: torch.Tensor, set_col: torch.Tensor, label_pos: torch.Tensor,
              weight: torch.Tensor, need_grad: bool = True):
    """Fused masked CE over T class sets (model/clip_tree.py:241-277).  Returns ``(loss [T], dlogits [B,U] | None)``."""
    lib = _cabi.load()
    logits = _require(logits, "logits", torch.float32)
    set_ptr = _require(set_ptr, "set_ptr", torch.int32)
    set_col = _require(set_col, "set_col", torch.int32)
    label_pos = _require(label_pos, "label_pos", torch.int32)
    weight = _require(weight, "weight", torch.float32)
    B, U = logits.shape
    T = label_pos.numel()
    loss = torch.empty((T,), dtype=torch.float32, device=logits.device)
    dl = torch.empty_like(logits) if need_grad else None
    nbytes = lib.hgr_masked_ce_workspace_bytes(B, U, T)
    # a buffer of its own: the scoring workspace's header carries state between scoring calls (hgr_score_topk)
    key = ("masked_ce", logits.device.index, _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            _retired.append(ws)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=logits.device)
        _workspaces[key] = ws
    _cabi.check(lib.hgr_masked_ce(_ptr(logits), logits.stride(0), B, U, _ptr(set_ptr), _ptr(set_col),
                                  _ptr(label_pos), _ptr(weight), T, _ptr(loss), _ptr(dl), _ptr(ws), ws.numel(),
                                  _stream()))
    return loss, dl


def om_backward(dlogits: torch.Tensor, logits: torch.Tensor, x: torch.Tensor, x_norm: torch.Tensor, tn: torch.Tensor,
                t_norm: torch.Tensor, scale: float, d_log_scale: Optional[torch.Tensor] = None):
    """Backward of ``logits = scale * x @ tn^T`` and of the two row normalisations (clip_tree.py:276 / :263 / :225,262 /
    :280) on the tcgen05 GEMM kernel.  Returns ``(d_img_raw [B,D] fp32, d_text_raw [U,D] fp32)``; ``d_log_scale``
    (fp32 [1], optional) is ACCUMULATED into."""
    lib = _cabi.load()
    dlogits = _require(dlogits, "dlogits", torch.float32)
    logits = _require(logits, "logits", torch.float32)
    x = _require(x, "x", torch.bfloat16)
    tn = _require(tn, "tn", torch.bfloat16)
    x_norm = _require(x_norm, "x_norm", torch.float32)
    t_norm = _require(t_norm, "t_norm", torch.float32)
    B, U = dlogits.shape
    D = x.shape[1]
    if logits.shape != dlogits.shape or x.shape[0] != B or tn.shape != (U, D):
        raise ValueError("om_backward: shapes disagree")
    d_img = torch.empty((B, D), dtype=torch.float32, device=x.device)
    d_text = torch.empty((U, D), dtype=torch.float32, device=x.device)
    nbytes = lib.hgr_om_backward_workspace_bytes(B, U, D)
    key = ("om_bwd", x.device.index, _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            _retired.append(ws)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        _workspaces[key] = ws
    _cabi.check(lib.hgr_om_backward(_ptr(dlogits), _ptr(logits), dlogits.stride(0), B, U, D, _ptr(x), _ptr(x_norm), _ptr(tn),
                                    _ptr(t_norm), float(scale), _ptr(d_img), _ptr(d_text), _ptr(d_log_scale), _ptr(ws),
                                    ws.numel(), _stream()))
    return d_img, d_text
