"""ctypes binding of libhgr_b200.so (include/hgr_b200.h).

The library is the product; there is no Python/torch fallback.  If the shared object is
missing, ``load()`` raises with the build command -- a GPU box must never silently run
something else.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HGR_LIB") or os.path.join(HERE, "lib", "libhgr_b200.so")   # HGR_LIB: kernel experiments

HGR_OK = 0
HGR_F32, HGR_BF16, HGR_F16 = 0, 1, 2
HGR_IMPL_AUTO, HGR_IMPL_SIMT, HGR_IMPL_TCGEN05 = 0, 1, 2
HGR_IMPL_TCGEN05_EXACT, HGR_IMPL_TCGEN05_NULL, HGR_IMPL_TCGEN05_SKETCH = 4, 5, 12
HGR_IMPL_FLAG_NO_MERGE = 0x100
HGR_IMPL_GRID_SHARE_SHIFT = 12
HGR_GRID_SHARE_MAX = 8
HGR_NUM_HITS = 5
HGR_TOPK_MAX = 32
HGR_HIER_MAX_CHAIN = 32
HGR_MAX_SPLITS = 8   # hgr_score_topk_splits: splits per call
HGR_MAX_GROUPS = 16  # ... and groups of equal split membership
HIT_CUTS = (1, 2, 5, 10, 20)  # main.py:120
HGR_MISTAKE_COUNTERS = 2 + 2 * HGR_NUM_HITS + 2 * HGR_HIER_MAX_CHAIN + 2   # hgr_hier_mistakes: counters per set

# every symbol include/hgr_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "hgr_version": (c_int, []),
    "hgr_last_error": (c_char_p, []),
    "hgr_launch_count": (c_int64, []),
    "hgr_aggregate_normalize": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                        c_int64, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
    "hgr_normalize_rows_dual": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgr_score_topk_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "hgr_score_topk_plan": (c_int, [c_int64, c_int64, c_int64, c_int, c_void_p]),
    "hgr_score_topk_footprint": (c_int, [c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "hgr_score_topk_plan_shared": (c_int, [c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "hgr_score_topk_grid_share": (c_int, [c_int64, c_int64, c_int64, c_int]),
    "hgr_score_topk_footprint_shared": (c_int, [c_int64, c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "hgr_score_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int64,
                               c_float, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_int,
                               c_void_p]),
    "hgr_topk_merge": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p]),
    "hgr_peer_alloc": (c_int, [c_size_t, c_void_p, c_void_p]),
    "hgr_peer_open": (c_int, [c_void_p, c_void_p]),
    "hgr_peer_close": (c_int, [c_void_p]),
    "hgr_peer_free": (c_int, [c_void_p]),
    "hgr_score_topk_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int64, c_int64, c_float, c_int,
                                       c_void_p, c_size_t, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "hgr_score_topk_global_list_len": (c_int, [c_int64, c_int64, c_int64, c_int, c_int64]),
    "hgr_score_topk_scatter_bounded": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int64, c_int64, c_float,
                                               c_int, c_void_p, c_size_t, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                               c_int64, c_int, c_void_p]),
    "hgr_topk_merge_certified": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_int64,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_float,
                                         c_void_p, c_void_p]),
    "hgr_sample_replay": (c_int64, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "hgr_sample_replay_many": (c_int64, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgr_om_plan": (c_int64, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgr_normalize_rows_bcast": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "hgr_peer_signal": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "hgr_peer_wait": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "hgr_logits_dense": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_float, c_void_p, c_int64,
                                 c_int, c_void_p]),
    "hgr_hier_metrics_fused_rows": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p,
                                            c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                            c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgr_score_topk_splits_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "hgr_score_topk_splits": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                      c_int64, c_float, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                      c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "hgr_hier_level_scatter": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int64, c_void_p,
                                       c_size_t, c_int64, c_int, c_void_p, c_void_p]),
    "hgr_hier_finish_rows_gathered": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p,
                                              c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                              c_void_p, c_void_p, c_void_p]),
    "hgr_score_topk_splits_scatter_bounded_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "hgr_score_topk_splits_global_list_len": (c_int, [c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int,
                                                      c_void_p]),
    "hgr_score_topk_splits_scatter_bounded": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int64, c_int64,
                                                      c_float, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                                      c_size_t, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                                      c_int, c_void_p]),
    "hgr_topk_merge_splits_certified": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int64,
                                                c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_int64, c_void_p, c_float, c_void_p, c_void_p]),
    "hgr_hier_mistakes": (c_int, [c_void_p, c_int64, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int64, c_void_p, c_void_p]),
    "hgr_class_hits": (c_int, [c_void_p, c_int64, c_int, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                               c_void_p]),
    "hgr_masked_ce_workspace_bytes":(c_size_t, [c_int64, c_int64, c_int64]),
    "hgr_om_backward_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "hgr_om_backward": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hgr_masked_ce": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
}

_lib = None


class HgrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libhgr_b200 error %d: %s" % (code, msg))
        self.code = code


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libhgr_b200.so is not built (%s).  Build it with `python -m hgrnet_b200.build` "
            "(needs nvcc; cross-compiles sm_100a without a GPU).  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != HGR_OK:
        raise HgrError(code, load().hgr_last_error().decode("utf-8", "replace"))


def launch_count() -> int:
    return int(load().hgr_launch_count())
