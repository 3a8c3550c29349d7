"""Class-sharded multi-GPU eval head (one process per GPU, ``torch.distributed`` / NCCL plumbing).

The reference is single-GPU (main.py:226).  Here the class bank is cut row-wise into ``G``
contiguous shards (SURVEY.md section 8e); every rank scores the WHOLE image batch against its shard
with the fused kernel (2), the per-rank ``[B, K]`` candidate lists (value, node id) are exchanged
with ONE ``all_gather`` per batch over NVLink, and every rank merges the ``G`` lists with
``hgr_topk_merge`` (which also counts Hit@k -- a label hit needs the GLOBAL rank, so hits cannot
be counted per shard).  No other collective is on the data path.

``ShardedScorer.score`` is synchronous; ``ShardedScorer.submit`` / ``collect`` pipeline batches so
that the all-gather + merge of batch i overlap the GEMM of batch i+1 (the exchange is latency
bound: 2*B*K*4 bytes per rank).

The production arrangement is ``ShardedEvalStream`` over ``PeerExchange`` / ``PeerBank``: no collective on the data
path -- every rank's scoring kernel stores its lists straight into the buffer of the rank that OWNS the image rows
(peer memory over NVLink, flag-ordered), the lists are narrow and sized for the row's GLOBAL stream, and the owner
certifies each row against the global K-th value (``hgr_score_topk_scatter_bounded`` / ``hgr_topk_merge_certified``),
repairing the rare uncertified row from the peers' bank shards.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import ops
from .evaluate import EvalCounters


def shard_bounds(C: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous row ranges ``[lo, hi)`` of ``ceil(C / world)`` rows (the last ones may be short or empty)."""
    per = (C + world - 1) // world
    return [(min(C, r * per), min(C, (r + 1) * per)) for r in range(world)]


def pack_candidates(val: torch.Tensor, idx: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One ``[2, B, K]`` int32 record per rank: fp32 value bits, then node ids -> a single all-gather."""
    if out is None:
        out = torch.empty((2,) + tuple(val.shape), dtype=torch.int32, device=val.device)
    out[0].copy_(val.view(torch.int32))
    out[1].copy_(idx)
    return out


def unpack_gathered(buf: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """``[G, 2, B, K]`` int32 -> strided ``[G, B, K]`` views (fp32 values, int32 ids), no copy."""
    return buf[:, 0].view(torch.float32), buf[:, 1]


class ShardedScorer:
    def __init__(self, bank_shard: torch.Tensor, col_id_shard: Optional[torch.Tensor], id_base: int = 0, K: int = 20,
                 group=None, depth: int = 2):
        self.bank = bank_shard
        self.col_id = col_id_shard
        self.id_base = id_base
        self.K = K
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.depth = depth
        self._slots = []          # per in-flight batch: (send buffer, gather buffer, work handle, targets, event)
        self._free = []
        self._merge_stream = None

    # ------------------------------------------------------------------ synchronous
    def score(self, x_norm: torch.Tensor, targets: Optional[torch.Tensor], hits: Optional[torch.Tensor] = None):
        self.submit(x_norm, targets)
        return self.collect(hits)

    # ------------------------------------------------------------------ pipelined
    def _buffers(self, B, device):
        while self._free:
            send, recv = self._free.pop()
            if send.shape[1] == B:
                return send, recv
        send = torch.empty((2, B, self.K), dtype=torch.int32, device=device)
        recv = torch.empty((self.world, 2, B, self.K), dtype=torch.int32, device=device)
        return send, recv

    def submit(self, x_norm: torch.Tensor, targets: Optional[torch.Tensor]):
        """Enqueue local scoring + the all-gather of one batch; returns immediately."""
        B = x_norm.shape[0]
        send, recv = self._buffers(B, x_norm.device)
        if self.bank.shape[0] > 0:
            val, idx = ops.score_topk(x_norm, self.bank, col_id=self.col_id, id_base=self.id_base, K=self.K)
        else:  # empty shard (more ranks than class chunks)
            val = torch.full((B, self.K), float("-inf"), device=x_norm.device)
            idx = torch.full((B, self.K), -1, dtype=torch.int32, device=x_norm.device)
        pack_candidates(val, idx, send)
        if self.world > 1:
            work = dist.all_gather_into_tensor(recv.view(-1), send.view(-1), group=self.group, async_op=True)
        else:
            recv[0].copy_(send)
            work = None
        self._slots.append((send, recv, work, targets))

    def collect(self, hits: Optional[torch.Tensor] = None):
        """Merge the oldest in-flight batch -> ``(val [B,K], idx [B,K])`` (+ hits)."""
        send, recv, work, targets = self._slots.pop(0)
        if work is not None:
            work.wait()  # orders the current stream after the collective; no host block
        pv, pi = unpack_gathered(recv)
        t = targets.to(torch.int32) if targets is not None else None
        out = ops.topk_merge(pv, pi, targets=t, hits=hits)
        self._free.append((send, recv))
        return out


class _RawCuda:
    """Zero-copy torch view of a raw device allocation (``torch.as_tensor`` reads ``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


X_SLOTS = 4  # feature-ingest slots per exchange (ring length per channel: _ring_len)


def exchange_layout(B: int, K: int, world: int, slots: int, D: int = 0, n_levels: int = 0, n_splits: int = 0):
    """Byte layout of one rank's exchange buffer: a 256-byte header (list flags: one word per producer rank at
    byte 0, feature flags at byte 64), then per slot the value lists ``[world, block_rows, K]`` fp32 followed by
    the id lists ``[world, block_rows, K]`` int32 and the bounds ``[world, block_rows]`` fp32 of the global certificate
    (``hgr_score_topk_scatter_bounded``) -- with ``n_splits`` one such area per split, ``split_bytes`` apart
    (``hgr_score_topk_splits_scatter_bounded``) --, with ``n_levels`` the per-level winner words ``[world, block_rows,
    n_levels]`` uint64 of class-sharded TOR / POR at ``hier_off`` in the slot (``hgr_hier_level_scatter``) and, when
    ``D`` is given, ``X_SLOTS`` replicas of the normalised image features ``[B, D]`` bf16 (feature ingest, see
    ``PeerExchange.ingest``)."""
    block_rows = (B + world - 1) // world
    part = block_rows * K * 4
    bound_bytes = (world * block_rows * 4 + 15) // 16 * 16     # per producer and row: bound of what the shard dropped
    slot_bytes = 2 * world * part + bound_bytes
    split = {}
    if n_splits:
        split = {"split_bytes": (slot_bytes + 15) // 16 * 16}  # every split's area 16-byte aligned
        slot_bytes = n_splits * split["split_bytes"]
    hier = {}
    if n_levels:
        # 8-byte aligned: both list areas are multiples of 8 bytes, the bounds of 16, and slots start 16-byte aligned
        hier = {"hier_off": slot_bytes, "hier_part_bytes": block_rows * n_levels * 8}
        slot_bytes = (slot_bytes + world * hier["hier_part_bytes"] + 15) // 16 * 16
    x_off = (256 + slots * slot_bytes + 255) // 256 * 256
    x_bytes = (B * D * 2 + 255) // 256 * 256
    return {"block_rows": block_rows, "part_bytes": part, "slot_bytes": slot_bytes, "header": 256,
            "x_off": x_off, "x_bytes": x_bytes, "total": x_off + (X_SLOTS * x_bytes if D else 0), **split, **hier}


class PeerMemoryUnavailable(RuntimeError):
    """Raised by ``PeerExchange`` on EVERY rank when any rank could not set the exchange up."""


def map_peer_buffers(nbytes: int, device, world: int, rank: int, group=None):
    """Allocate ``nbytes`` of zeroed device memory on this rank (``hgr_peer_alloc``), swap the CUDA IPC handles through
    ``torch.distributed`` and map every peer's allocation -> ``(own pointer, [pointer of rank g's buffer], [mapped])``.
    A failure on ANY rank (no CUDA IPC in the container, no peer access between two GPUs, out of memory) is agreed on
    collectively: every rank frees what it holds and raises ``PeerMemoryUnavailable``, so that callers can fall back
    together (the NCCL exchange) instead of deadlocking in the next collective."""
    err = None
    own, handle = None, None
    opened = []

    def release():
        for p in opened:
            ops.peer_close(p)
        if own is not None:
            ops.peer_free(own)

    with torch.cuda.device(device):
        try:
            own, handle = ops.peer_alloc(nbytes)
        except Exception as e:  # noqa: BLE001 -- reported through the agreement below
            err = e
        if world == 1:
            if err is not None:
                raise PeerMemoryUnavailable("peer_alloc failed: %r" % (err,))
            return own, [own], opened
        handles = [None] * world
        dist.all_gather_object(handles, handle, group=group)
        bases = []
        if err is None and all(h is not None for h in handles):
            try:
                for g in range(world):
                    if g == rank:
                        bases.append(own)
                    else:
                        bases.append(ops.peer_open(handles[g]))
                        opened.append(bases[-1])
            except Exception as e:  # noqa: BLE001
                err = e
        elif err is None:
            err = RuntimeError("a peer could not allocate its exchange buffer")
        oks = [None] * world
        dist.all_gather_object(oks, err is None, group=group)
        if not all(oks):
            release()
            raise PeerMemoryUnavailable("peer-memory exchange unavailable on rank(s) %s%s" % (
                [g for g, ok in enumerate(oks) if not ok], "" if err is None else ": %r" % (err,)))
        return own, bases, opened


class PeerBank:
    """A rank's class-bank shard (+ its node ids) in peer-visible memory, and the ``hgr_shard_t`` table of ALL ranks'
    shards: what the owner of an image row needs to repair a row whose global certificate failed
    (``hgr_topk_merge_certified`` re-scans the doubtful shard, over NVLink when it is a peer's)."""

    def __init__(self, bank_shard: torch.Tensor, col_id: Optional[torch.Tensor], id_base: int, group=None):
        self.device = bank_shard.device
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        C, D = bank_shard.shape
        bank_bytes = (C * D * 2 + 255) // 256 * 256
        nbytes = max(256, bank_bytes + (C * 4 if col_id is not None else 0))
        self._own, bases, self._opened = map_peer_buffers(nbytes, self.device, world, rank, group)
        raw = torch.as_tensor(_RawCuda(self._own, nbytes), device=self.device)
        self.bank = raw[:C * D * 2].view(torch.bfloat16).view(C, D)
        self.bank.copy_(bank_shard)
        self.col_id = None
        if col_id is not None:
            self.col_id = raw[bank_bytes:bank_bytes + C * 4].view(torch.int32)
            self.col_id.copy_(col_id)
        meta = [None] * world
        mine = (C, bank_bytes if col_id is not None else -1, int(id_base))
        if world > 1:
            dist.all_gather_object(meta, mine, group=group)
        else:
            meta = [mine]
        self.table = ops.shard_table([(bases[g], bases[g] + meta[g][1] if meta[g][1] >= 0 else 0, meta[g][0], meta[g][2])
                                      for g in range(world)], self.device)
        self.C_total = sum(m[0] for m in meta)
        torch.cuda.synchronize(self.device)
        if world > 1:
            dist.barrier(group=group)          # every shard is in place before anybody may re-scan it

    def close(self) -> None:
        for p in self._opened:
            ops.peer_close(p)
        self._opened = []
        if self._own is not None:
            ops.peer_free(self._own)
            self._own = None


class HierShard:
    """One rank's part of class-sharded TOR / POR (main.py:143,152-191): its contiguous slice ``[row_base, row_base +
    M_r)`` of the level-sorted train bank (``shard_bounds`` over the sorted rows, so the GEMM columns are balanced) with
    the global level ends clipped to it, and the global tables the row owner needs to finish its rows.  ``rows_args`` is
    what ``evaluate.HierMetrics.rows_args()`` returns."""

    def __init__(self, rows_args: dict, rank: int, world: int):
        bank = rows_args["bank_sorted"]
        self.M, self.D = bank.shape
        self.level_end = [int(e) for e in rows_args["level_end"]]
        self.n_levels = len(self.level_end)
        if not 1 <= self.n_levels <= 32:
            raise ValueError("class-sharded TOR / POR supports 1 to 32 levels, got %d" % self.n_levels)
        lo, hi = shard_bounds(self.M, world)[rank]
        self.row_base = lo
        self.bank = bank[lo:hi]                  # a row slice of a contiguous tensor: contiguous, 16-byte aligned
        self.level_end_local = local_level_ends(self.level_end, lo, hi)
        self.sorted_to_pos, self.first_out = rows_args["sorted_to_pos"], rows_args["first_out"]
        self.chain_ptr, self.chain_pos, self.chain_level = (rows_args["chain_ptr"], rows_args["chain_pos"],
                                                            rows_args["chain_level"])


def local_level_ends(level_end, lo: int, hi: int) -> List[int]:
    """The global level ends of the sorted train bank clipped to the shard ``[lo, hi)``: non-decreasing, ending at
    ``hi - lo``."""
    return [min(max(int(e) - lo, 0), hi - lo) for e in level_end]


def split_shard_bounds(group_end, world: int):
    """How the union bank of ``evaluate.split_groups`` is cut over ``world`` ranks: every rank takes its balanced slice
    ``[floor(r * C_g / world), floor((r + 1) * C_g / world))`` of EVERY group g, so it holds about 1/world of every
    split (a contiguous cut would leave a small split on one or two ranks).  Returns, per rank, ``(ranges, local_end,
    kept)``: the union-bank row ranges ``[lo, hi)`` of the groups it holds rows of (``kept``, ascending), concatenated in
    that order its local bank, and their clipped ends ``local_end`` (strictly ascending: groups without rows here are
    dropped).  A rank may hold no rows at all."""
    out = []
    begins = [0] + [int(e) for e in group_end[:-1]]
    for r in range(world):
        ranges, local_end, kept, n = [], [], [], 0
        for g, (b, e) in enumerate(zip(begins, [int(e) for e in group_end])):
            lo, hi = b + (e - b) * r // world, b + (e - b) * (r + 1) // world
            if hi > lo:
                ranges.append((lo, hi))
                n += hi - lo
                local_end.append(n)
                kept.append(g)
        out.append((ranges, local_end, kept))
    return out


class SplitShard:
    """One rank's part of several test splits scored in one pass on the class-sharded head (main.py:104-222 once per
    split): its slice of every group of ``split_eval``'s union bank (``split_shard_bounds``) with its node ids
    (``col_id``), its own group table (``group_end`` / ``group_splits``, the masks of the groups it holds), the global
    class count of every split (``split_C``) and ``node_splits`` / ``names`` / ``S``.  With ``split_eval.hier`` it also
    holds the rank's ``HierShard`` of the level-sorted train bank (per-split TOR / POR).  ``split_eval`` is an
    ``evaluate.SplitEval`` (or anything with its ``group_end``, ``group_splits``, ``names``, ``S``, ``node_splits``,
    ``col_id``, ``bank()`` and ``hier``)."""

    def __init__(self, split_eval, rank: int, world: int):
        ranges, self.group_end, kept = split_shard_bounds(split_eval.group_end, world)[rank]
        union = split_eval.bank()
        self.device = union.device
        rows = (torch.cat([torch.arange(lo, hi) for lo, hi in ranges]) if ranges
                else torch.zeros(0, dtype=torch.int64)).to(self.device)
        self.bank = union.index_select(0, rows).contiguous()
        self.col_id = split_eval.col_id.index_select(0, rows).to(torch.int32).contiguous()
        self.C, self.D = self.bank.shape
        self.group_splits = [int(split_eval.group_splits[g]) for g in kept]
        self.names, self.S = list(split_eval.names), int(split_eval.S)
        self.node_splits = split_eval.node_splits
        ends = [int(e) for e in split_eval.group_end]
        sizes = [e - b for b, e in zip([0] + ends[:-1], ends)]
        self.split_C = [sum(n for n, m in zip(sizes, split_eval.group_splits) if (int(m) >> s) & 1) for s in range(self.S)]
        h = getattr(split_eval, "hier", None)
        self.hier = HierShard(h.rows_args(), rank, world) if h is not None else None


class MistakeShard:
    """One rank's part of the class-sharded mistake severity and LCA distance@k (``evaluate.MistakeMetrics``): the
    chain table, which every rank holds whole, and the image rows this rank owns and counts.  The owner runs
    ``ops.hier_mistakes`` on its merged lists, so nothing of it crosses the exchange.  ``rank`` / ``world`` default to
    the process group's."""

    def __init__(self, mistakes, rank: Optional[int] = None, world: Optional[int] = None, group=None):
        if world is None:
            world = dist.get_world_size(group) if dist.is_initialized() else 1
        if rank is None:
            rank = dist.get_rank(group) if dist.is_initialized() else 0
        if not 0 <= rank < world:
            raise ValueError("rank %d outside [0, %d)" % (rank, world))
        self.rank, self.world = rank, world
        self.chain_ptr, self.chain_node = mistakes.chain_ptr, mistakes.chain_node

    def args(self) -> dict:
        return dict(chain_ptr=self.chain_ptr, chain_node=self.chain_node)

    def row_bounds(self, B: int) -> Tuple[int, int]:
        """The rows ``[lo, hi)`` of a batch of ``B`` this rank owns, merges and counts (``PeerExchange``'s blocks)."""
        block_rows = (B + self.world - 1) // self.world
        lo = min(B, self.rank * block_rows)
        return lo, min(B, lo + block_rows)


class PeerExchange:
    """Peer-memory exchange of the class-sharded head (no collective call on the data path).

    Rank ``g`` owns image rows ``[g * block_rows, (g + 1) * block_rows)``.  Every rank allocates one exchange buffer
    (``hgr_peer_alloc``), the CUDA IPC handles are swapped once through ``torch.distributed`` and every peer buffer
    is mapped into this process (``hgr_peer_open``).  Per batch a rank's scoring kernel then writes its local top-K
    of row block ``g`` directly into list ``rank`` of rank ``g``'s buffer over NVLink (``hgr_score_topk_scatter``)
    and raises its flag there (``hgr_peer_signal``); the owner waits for all ``world`` flags (``hgr_peer_wait``) and
    merges its ``world`` lists per row (``hgr_topk_merge``).  ``slots`` batches can be in flight.  With ``n_levels``
    every slot also carries the per-level winner words of class-sharded TOR / POR (``scatter`` / ``merge`` with
    ``hier``), published by the same flag.  With ``n_splits`` every slot holds the lists and bounds of that many test
    splits (``scatter`` / ``merge`` with ``splits``).
    """

    def __init__(self, B: int, K: int, device, group=None, slots: int = 4, D: int = 0, _bases=None, _rank=None,
                 _world=None, n_levels: int = 0, n_splits: int = 0):
        self.device = torch.device(device)
        self.group = group
        if _bases is None:
            self.world = dist.get_world_size(group) if dist.is_initialized() else 1
            self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        else:                                  # several logical ranks inside one process (single-GPU tests)
            self.world, self.rank = _world, _rank
        if self.world > 16:
            raise ValueError("PeerExchange supports up to 16 ranks (HGR_MAX_PEERS)")
        self.B, self.K, self.slots, self.D, self.n_levels = B, K, slots, D, n_levels
        self.lay = exchange_layout(B, K, self.world, slots, D, n_levels, n_splits)
        self.split_stride = self.lay.get("split_bytes", 0) // 4     # elements between two splits' areas
        self.block_rows = self.lay["block_rows"]
        self.lo = min(B, self.rank * self.block_rows)
        self.hi = min(B, self.lo + self.block_rows)
        self._opened = []
        if _bases is not None:
            self.bases = list(_bases)
            self._own = None
        else:
            self._own = None
            self._map_peers(group)
        self.local = torch.as_tensor(_RawCuda(self.bases[self.rank], self.lay["total"]), device=self.device)
        self.seq = torch.zeros(4, dtype=torch.int32, device=self.device)   # lists: [sent, waited]; features: same
        self.flag_ptrs = [b + 4 * self.rank for b in self.bases]
        self.xflag_ptrs = [b + 64 + 4 * self.rank for b in self.bases]

    def _map_peers(self, group) -> None:
        self._own, self.bases, self._opened = map_peer_buffers(self.lay["total"], self.device, self.world, self.rank, group)

    # -- addresses -------------------------------------------------------------------------------------------
    def _slot_base(self, base: int, slot: int) -> int:
        return base + self.lay["header"] + slot * self.lay["slot_bytes"]

    def block_ptrs(self, slot: int):
        """Where THIS rank's lists of row block g go: list ``rank`` of rank g's slot."""
        part, world = self.lay["part_bytes"], self.world
        val = [self._slot_base(b, slot) + self.rank * part for b in self.bases]
        idx = [self._slot_base(b, slot) + world * part + self.rank * part for b in self.bases]
        return val, idx

    def bound_ptrs(self, slot: int):
        """Where THIS rank's bounds of row block g go: row ``rank`` of the bound area of rank g's slot."""
        off = 2 * self.world * self.lay["part_bytes"] + self.rank * self.block_rows * 4
        return [self._slot_base(b, slot) + off for b in self.bases]

    def local_bounds(self, slot: int) -> int:
        """Pointer to the ``[world, block_rows]`` bounds received for my rows."""
        return self._slot_base(self.bases[self.rank], slot) + 2 * self.world * self.lay["part_bytes"]

    def local_parts(self, slot: int):
        """(value pointer, id pointer, element stride) of the ``world`` lists received for my rows."""
        base = self._slot_base(self.bases[self.rank], slot)
        return base, base + self.world * self.lay["part_bytes"], self.block_rows * self.K

    def hier_ptrs(self, slot: int):
        """Where THIS rank's winner words of row block g go: region ``rank`` of the TOR / POR area of rank g's slot."""
        off = self.lay["hier_off"] + self.rank * self.lay["hier_part_bytes"]
        return [self._slot_base(b, slot) + off for b in self.bases]

    def local_hier(self, slot: int):
        """(pointer, word stride) of the ``world`` winner-word arrays received for my rows."""
        return self._slot_base(self.bases[self.rank], slot) + self.lay["hier_off"], self.block_rows * self.n_levels

    # -- feature ingest ----------------------------------------------------------------------------------------
    def x_ptrs(self, xslot: int):
        return [b + self.lay["x_off"] + xslot * self.lay["x_bytes"] for b in self.bases]

    def x_view(self, xslot: int) -> torch.Tensor:
        """The local replica of the normalised features of a slot, ``[B, D]`` bf16."""
        off = self.lay["x_off"] + xslot * self.lay["x_bytes"]
        return self.local[off:off + self.B * self.D * 2].view(torch.bfloat16).view(self.B, self.D)

    def ingest(self, feats_block: torch.Tensor, xslot: int) -> torch.Tensor:
        """``feats_block``: MY rows ``[hi - lo, D]`` of the batch (any float dtype).  Normalises them, stores them
        into every rank's replica over NVLink, waits until all ``world`` blocks have arrived here and returns the
        complete normalised batch ``[B, D]`` bf16 (a view of the exchange buffer)."""
        if not self.D:
            raise ValueError("PeerExchange was built without a feature area (D = 0)")
        if self.hi > self.lo:
            ops.normalize_rows_bcast(feats_block, self.lo, self.x_ptrs(xslot))
        ops.peer_signal(self.xflag_ptrs, self.seq[2:3])
        ops.peer_wait(self.bases[self.rank] + 64, self.world, self.seq[3:4])
        return self.x_view(xslot)

    # -- per batch -------------------------------------------------------------------------------------------
    def scatter(self, x_norm: torch.Tensor, bank: torch.Tensor, id_base: int, slot: int, col_id=None,
                C_total: int = 0, hier: Optional[HierShard] = None, splits: Optional[SplitShard] = None) -> None:
        """Score the batch against my shard and store the lists at their owners.  ``C_total`` > 0: narrow lists sized
        for the GLOBAL certificate, with the bound of what was dropped next to every list (``merge(certify=...)``).
        ``hier``: also store my train shard's per-level winner words at the owners (``merge(hier=...)``).  ``splits``:
        ``bank`` / ``col_id`` are my part of the split union bank; every split's lists and bounds are stored
        (``merge(splits=...)``)."""
        val, idx = self.block_ptrs(slot)
        if splits is not None:
            ops.score_topk_splits_scatter(x_norm, bank, splits.group_end, splits.group_splits, splits.split_C, val, idx,
                                          self.bound_ptrs(slot), self.block_rows, self.split_stride, col_id=col_id,
                                          K=self.K)
        else:
            ops.score_topk_scatter(x_norm, bank, val, idx, self.block_rows, col_id=col_id, id_base=id_base, K=self.K,
                                   bound_block_ptrs=self.bound_ptrs(slot) if C_total else None, C_total=C_total)
        if hier is not None:                 # before the signal: the owner's one wait covers lists and words
            ops.hier_level_scatter(x_norm, hier.bank, hier.level_end_local, hier.row_base, self.hier_ptrs(slot),
                                   self.block_rows)
        ops.peer_signal(self.flag_ptrs, self.seq[0:1])

    def merge(self, slot: int, targets: Optional[torch.Tensor], hits: Optional[torch.Tensor], out=None,
              targets_local: bool = False, certify=None, hier: Optional[HierShard] = None,
              counts: Optional[torch.Tensor] = None, hier_out=None, splits: Optional[SplitShard] = None,
              split_counts: Optional[torch.Tensor] = None):
        """Final top-K (+ hits) of MY rows ``[lo, hi)``; ``targets`` holds the labels of the whole batch (or of my
        rows only with ``targets_local``).  ``certify = (x_norm [B, D], shard table, repair counter)`` after a
        ``scatter(C_total=...)``: rows whose K-th value does not beat every shard's bound are repaired exactly.
        ``hier`` after a ``scatter(hier=...)``: also count TOR / POR of my rows into ``counts`` (``ops.new_hier_counts``);
        ``hier_out = (lvl_idx [n, n_levels], top1 [n])`` int32 receives their per-level winners and top-1.
        ``splits`` after a ``scatter(splits=...)`` (needs ``certify``): per split the certified top-K of my rows
        (``[S, n, K]``), Hit@k and rows counted into ``split_counts`` ``[S, HGR_NUM_HITS + 1]``; with ``hier``, ``counts``
        holds the per-split TOR / POR counters ``[S, HGR_HIER_MAX_CHAIN + 1, 4]`` (``ops.new_hier_counts(device, S)``)."""
        ops.peer_wait(self.bases[self.rank], self.world, self.seq[1:2])
        n = self.hi - self.lo
        if n <= 0:
            return None
        pv, pi, stride = self.local_parts(slot)
        t = None if targets is None else (targets if targets_local else targets[self.lo:self.hi])
        if splits is not None:
            x_norm, table, repairs = certify
            res = ops.topk_merge_splits_certified(pv, pi, self.local_bounds(slot), self.world, n, self.K, splits.S, stride,
                                                  self.block_rows, self.split_stride, x_norm[self.lo:self.hi], table,
                                                  splits.node_splits, self.device, targets=t, counts=split_counts,
                                                  repair_count=repairs, out=out)
        elif certify is not None:
            x_norm, table, repairs = certify
            res = ops.topk_merge_certified(pv, pi, self.local_bounds(slot), self.world, n, self.K, stride, self.block_rows,
                                           x_norm[self.lo:self.hi], table, self.device, targets=t, hits=hits,
                                           repair_count=repairs, out=out)
        else:
            res = ops.topk_merge_raw(pv, pi, self.world, n, self.K, stride, self.device, targets=t, hits=hits, out=out)
        if hier is not None:
            parts, part_stride = self.local_hier(slot)
            lvl_idx, top1 = hier_out if hier_out is not None else (None, None)
            ops.hier_finish_rows_gathered(parts, self.world, part_stride, n, hier.M, hier.n_levels, hier.sorted_to_pos,
                                          hier.first_out, t, hier.chain_ptr, hier.chain_pos, hier.chain_level, counts,
                                          node_splits=None if splits is None else splits.node_splits, lvl_idx=lvl_idx,
                                          top1=top1)
        return res

    def close(self) -> None:
        for p in self._opened:
            ops.peer_close(p)
        self._opened = []
        if self._own is not None:
            ops.peer_free(self._own)
            self._own = None


def _ring_len(n_c: int, slots: int) -> int:
    """Ring length <= slots for a channel that runs n_c >= 2 batches per replay: consecutive batches, including the
    last one of a replay and the first one of the next, must use different slots: (n_c - 1) % ring != 0."""
    for ring in range(slots, 1, -1):
        if (n_c - 1) % ring != 0:
            return ring
    raise ValueError("no safe slot ring for %d batches per channel" % n_c)


class ShardedEvalStream:
    """Software-pipelined, CUDA-graph captured class-sharded eval steps (one process per GPU).

    One graph holds ``steps`` consecutive batches.  Two exchanges:

    * ``exchange="p2p"`` (default): ``PeerExchange`` -- the scoring kernel's final lists go straight into the row
      owner's buffer over NVLink, a flag word per producer orders them; the owner merges ITS rows only (1/world of
      the merge work, 1/world of the bytes of an all-gather, no collective kernel competing for SMs).  The merge of
      batch i is issued after the scoring of batch i+1, so the flags have long arrived when it runs.  Results
      (``val`` / ``idx``) cover rows ``[row_lo, row_hi)``; ``hits`` counts those rows -- sum it over ranks at the end
      (``all_reduce_hits``: the one collective of an evaluation).
    * ``exchange="nccl"``: ``normalise -> score -> all_gather_into_tensor`` (NCCL stream) ``-> merge`` of all rows
      on every rank, the gather of batch i overlapping the GEMM of batch i+1.

    A replay is one ``cudaGraphLaunch`` for ``steps`` batches: no interpreter, no per-batch launch latency.

    ``hier`` (a ``HierShard`` of this rank, peer exchange only): every batch also counts TOR / POR (main.py:143,152-191)
    of the rows this rank owns, against each row's own label.  The rank's slice of the level-sorted train bank runs the
    per-level arg-max GEMM, its winner words travel to the row owners with the lists, under the same flag, and the owner
    finishes its rows after the list merge.  The per-chain-length counters share one device buffer with ``hits``
    (``counters``), so ``host_io`` still makes one D2H copy per batch; ``hier_ratios()`` sums them over ranks.

    ``splits`` (a ``SplitShard`` of this rank, peer exchange with the global certificate only): every batch is scored
    against the rank's part of several test splits instead of ``bank_shard``, in one pass, as ``EvalStream(splits=...)``
    does on one GPU.  ``val`` / ``idx`` are ``[S, rows, K]``; the per-split Hit@k / row counters ``split_counts``
    ``[S, HGR_NUM_HITS + 1]`` and, when the ``SplitShard`` has ``hier``, the per-split TOR / POR counters
    ``hier_counts`` ``[S, HGR_HIER_MAX_CHAIN + 1, 4]`` live in ``counters`` too.  ``split_hit_counts()`` /
    ``split_ratios()`` / ``split_lines()`` sum them over ranks.  With ``splits`` the stream scores nothing against
    ``bank_shard`` / ``id_base``: ``bank_shard`` only has to agree with the ``SplitShard`` on D and device (pass e.g.
    ``split_eval.bank()``), and ``id_base`` is unused.

    ``mistakes`` (a ``MistakeShard`` of this rank, peer exchange only, with or without ``splits``): after the merge the
    row owner counts the mistake severity and LCA distance@k of its merged lists against each row's own label
    (``ops.hier_mistakes``; one counter set per split with ``splits``).  No exchange data and no flag is added; the
    counters sit in ``counters``, and ``mistake_summary()`` / ``split_mistake_summary()`` sum them over ranks.

    ``classes`` (an ``evaluate.ClassHits``, peer exchange only, with or without ``splits``): after the merge the row
    owner counts Hit@k per class of its merged lists against each row's own label (``ops.class_hits``; one table per
    split with ``splits``).  No exchange data and no flag is added.  The table is a device buffer of its own
    (``class_counts``), outside ``counters``, so the per-batch ``host_counters`` copy keeps its size; ``class_table()`` /
    ``class_summary()`` / ``split_class_summary()`` sum it over ranks.
    """

    def __init__(self, bank_shard: torch.Tensor, id_base: int, *, batch: int, K: int = 20, steps: int = 8,
                 feat_dtype=torch.float32, banks=None, group=None, use_graph: bool = True, exchange: str = "p2p",
                 channels: int = 4, host_io: bool = False, col_id: Optional[torch.Tensor] = None,
                 certify: str = "global", hier: Optional[HierShard] = None, splits: Optional[SplitShard] = None,
                 mistakes: Optional[MistakeShard] = None, classes=None):
        if exchange not in ("p2p", "nccl"):
            raise ValueError("exchange must be 'p2p' or 'nccl'")
        if splits is not None:
            if exchange != "p2p":
                raise ValueError("splits need the peer-memory exchange")
            if certify != "global":
                raise ValueError("splits need certify='global'")
            if hier is not None:
                raise ValueError("splits and hier together: the splits' TOR / POR come with the SplitShard's hier")
            if banks is not None:
                raise ValueError("splits do not take a banks= rotation")
            if splits.D != bank_shard.shape[1] or splits.device != bank_shard.device:
                raise ValueError("splits: the SplitShard has D = %d on %s, the stream D = %d on %s" % (
                    splits.D, splits.device, bank_shard.shape[1], bank_shard.device))
        if mistakes is not None:
            if exchange != "p2p":
                raise ValueError("mistakes (class-sharded mistake metrics) need the peer-memory exchange")
            if mistakes.chain_ptr.device != bank_shard.device:
                raise ValueError("mistakes: the chain table is on %s, the bank on %s" % (mistakes.chain_ptr.device,
                                                                                       bank_shard.device))
        if classes is not None:
            if exchange != "p2p":
                raise ValueError("classes (class-sharded per-class Hit@k) need the peer-memory exchange")
            if classes.counts.device != bank_shard.device:
                raise ValueError("classes: the counters are on %s, the bank on %s" % (classes.counts.device,
                                                                                    bank_shard.device))
        if hier is not None and exchange != "p2p":
            raise ValueError("hier (class-sharded TOR / POR) needs the peer-memory exchange")
        if hier is not None and hier.D != bank_shard.shape[1]:
            raise ValueError("hier: the train bank has D = %d, the class bank %d" % (hier.D, bank_shard.shape[1]))
        if certify not in ("global", "local"):
            raise ValueError("certify must be 'global' or 'local'")
        if host_io and exchange != "p2p":
            raise ValueError("host_io needs the peer-memory exchange")
        self.exchange, self.host_io = exchange, host_io
        self.device = bank_shard.device
        self.banks = list(banks) if banks is not None else [bank_shard]
        self.id_base, self.K, self.B, self.steps, self.group = id_base, K, batch, steps, group
        self.col_id = col_id          # node id of every bank row of this shard (None: id_base + row)
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        D = bank_shard.shape[1]
        # certify="global" (peer exchange only): the lists a rank keeps are sized for the row's GLOBAL stream and
        # certified by the owner of the row against the global K-th value (hgr_score_topk_scatter_bounded /
        # hgr_topk_merge_certified) -- a shard's own stream is too short for narrow lists to be certified locally, and
        # exact 20-entry lists cost 39 us instead of 27 per call at the N = 8 shard.  The owner repairs an uncertified
        # row by re-scanning the doubtful shard, so every rank's shard lives in peer-visible memory (PeerBank).
        self.certify = certify if exchange == "p2p" else "local"
        self.C_total = 0
        self.repairs = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._x = [None] * steps
        self.splits = splits
        if splits is not None:
            self.banks, col_id, self.id_base = [splits.bank], splits.col_id, 0
        if self.certify == "global":
            self.pbanks = [PeerBank(b, col_id, self.id_base, group) for b in self.banks]
            self.banks = [pb.bank for pb in self.pbanks]
            self.col_id = self.pbanks[0].col_id
            self.C_total = self.pbanks[0].C_total
        if not host_io:
            self.dev_feats = [torch.empty((batch, D), dtype=feat_dtype, device=self.device) for _ in range(steps)]
            self.dev_labels = [torch.zeros((batch,), dtype=torch.int32, device=self.device) for _ in range(steps)]
        # every counter of the stream in one device buffer (evaluate.EvalCounters): one D2H copy per batch
        self.hier = hier
        S = 0 if splits is None else splits.S
        self.mistakes = mistakes
        self.tally = EvalCounters(self.device, n_splits=S, hier=self._hier_shard() is not None,
                                  mistakes=mistakes is not None, K=K, read=self._read_counters,
                                  classes=0 if classes is None else classes.n_nodes)
        self.counters, self.hits = self.tally.counters, self.tally.hits
        self.split_counts, self.hier_counts = self.tally.split_counts, self.tally.hier_counts
        self.mistake_counts = self.tally.mistake_counts
        self.class_counts = self.tally.class_counts
        n_counters = self.counters.numel()
        self.val = [None] * steps
        self.idx = [None] * steps
        self.row_lo, self.row_hi = 0, batch
        if exchange == "p2p":
            self.slots = 4
            # `channels` independent exchanges (own flags, counters, slots), one CUDA stream each: batch s runs on
            # channel s % channels, so the normalise / merge kernels of one batch fill the SMs the persistent GEMM
            # of the neighbouring batch leaves idle at its edges
            # Slot reuse: a producer may overwrite a list slot of batch j once the owner has merged batch j, which it
            # knows from the owner's NEXT signal -- so two consecutive batches of a channel must never share a slot,
            # also across the replay boundary (a replay restarts at slot 0).  Every channel therefore gets at least two
            # batches per replay and a ring length `_ring[c]` that its batch count does not wrap onto itself with.
            if steps < 2:
                raise ValueError("ShardedEvalStream needs steps >= 2 (two batches per exchange channel and replay)")
            self.channels = max(1, min(channels, steps // 2))
            hs = self._hier_shard()
            self.pxs = [PeerExchange(batch, K, self.device, group=group, slots=self.slots, D=D if host_io else 0,
                                     n_levels=0 if hs is None else hs.n_levels, n_splits=S)
                        for _ in range(self.channels)]
            self._ring, self._xring = [], []
            for c in range(self.channels):
                n_c = (steps - c + self.channels - 1) // self.channels          # batches of channel c per replay
                self._ring.append(_ring_len(n_c, self.slots))
                self._xring.append(_ring_len(n_c, X_SLOTS))
            self.px = self.pxs[0]
            self.side = [torch.cuda.Stream(device=self.device) for _ in range(self.channels)]
            self.row_lo, self.row_hi = self.px.lo, self.px.hi
            n_my = max(0, self.row_hi - self.row_lo)
            shape = (n_my, K) if splits is None else (S, n_my, K)
            self.val = [torch.empty(shape, dtype=torch.float32, device=self.device) for _ in range(steps)]
            self.idx = [torch.empty(shape, dtype=torch.int32, device=self.device) for _ in range(steps)]
            if host_io:
                # feature ingest: this rank copies only ITS rows (and their labels) from pinned host memory; the
                # normalised rows reach the other ranks over NVLink (PeerExchange.ingest); Hit@k counters go back
                # to the host after every batch
                # (features + labels of a batch share one staging buffer per side: a single DMA per batch)
                fbytes = n_my * D * torch.empty((), dtype=feat_dtype).element_size()

                def views(pack):
                    return pack[:fbytes].view(feat_dtype).view(n_my, D), pack[fbytes:].view(torch.int32)

                self.host_pack = [torch.zeros(fbytes + n_my * 4, dtype=torch.uint8, pin_memory=True) for _ in range(steps)]
                self.dev_pack = [torch.zeros(fbytes + n_my * 4, dtype=torch.uint8, device=self.device) for _ in range(steps)]
                self.host_feats, self.host_labels = map(list, zip(*[views(p) for p in self.host_pack]))
                self.dev_feats, self.dev_labels = map(list, zip(*[views(p) for p in self.dev_pack]))
                self.host_counters = [torch.zeros((n_counters,), dtype=torch.int64, pin_memory=True)
                                      for _ in range(steps)]
                self.host_hits = [c[:ops.HGR_NUM_HITS] for c in self.host_counters]
            if self.world > 1:
                dist.barrier(group=group)          # every buffer is mapped everywhere before the first store
        else:
            self.send = [torch.empty((2, batch, K), dtype=torch.int32, device=self.device) for _ in range(steps)]
            self.recv = [torch.empty((self.world, 2, batch, K), dtype=torch.int32, device=self.device)
                         for _ in range(steps)]
        self.graph = None
        self.stream = torch.cuda.Stream(device=self.device)
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.stream):
            self._issue()                      # warm-up: NCCL communicator, workspaces
            self.stream.synchronize()
            self.tally.zero_()
            if use_graph:
                try:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=self.stream):
                        self._issue()
                    self.graph = g
                except Exception as e:  # pragma: no cover - depends on the NCCL / torch build
                    print("ShardedEvalStream: graph capture of the NCCL pipeline failed (%r); running eagerly" % (e,))
                    self.graph = None
        torch.cuda.synchronize(self.device)
        self.tally.zero_()

    def _local(self, s: int):
        bank = self.banks[s % len(self.banks)]
        if self.host_io:
            px, j = self.pxs[s % self.channels], s // self.channels
            self.dev_pack[s].copy_(self.host_pack[s], non_blocking=True)
            x = px.ingest(self.dev_feats[s], j % self._xring[s % self.channels])
            self._x[s] = x
            px.scatter(x, bank, self.id_base, j % self._ring[s % self.channels], col_id=self.col_id, C_total=self.C_total,
                       hier=self._hier_shard(), splits=self.splits)
            return None
        x = ops.normalize_rows(self.dev_feats[s])
        if self.exchange == "p2p":
            self._x[s] = x           # the owner's repair reads the row's features (kept alive for the captured graph)
            self.pxs[s % self.channels].scatter(x, bank, self.id_base, (s // self.channels) % self._ring[s % self.channels],
                                                col_id=self.col_id, C_total=self.C_total, hier=self._hier_shard(),
                                                splits=self.splits)
            return None
        if bank.shape[0] > 0:
            # results go straight into the send record (no pack copies)
            ops.score_topk(x, bank, col_id=self.col_id, id_base=self.id_base, K=self.K,
                           out=(self.send[s][0].view(torch.float32), self.send[s][1]))
        else:
            self.send[s][0].copy_(torch.full((self.B, self.K), float("-inf"), device=self.device).view(torch.int32))
            self.send[s][1].fill_(-1)
        if self.world > 1:
            return dist.all_gather_into_tensor(self.recv[s].view(-1), self.send[s].view(-1), group=self.group,
                                               async_op=True)
        self.recv[s][0].copy_(self.send[s])
        return None

    def _merge(self, s: int, work):
        if self.exchange == "p2p":
            cert = None
            if self.certify == "global":
                cert = (self._x[s], self.pbanks[s % len(self.pbanks)].table, self.repairs)
            self.pxs[s % self.channels].merge((s // self.channels) % self._ring[s % self.channels], self.dev_labels[s], self.hits,
                                              out=(self.val[s], self.idx[s]), targets_local=self.host_io, certify=cert,
                                              hier=self._hier_shard(), counts=self.hier_counts, splits=self.splits,
                                              split_counts=self.split_counts)
            t = self.dev_labels[s] if self.host_io else self.dev_labels[s][self.row_lo:self.row_hi]
            node_splits = None if self.splits is None else self.splits.node_splits
            if self.mistakes is not None and self.row_hi > self.row_lo:     # the owner's merged lists, after the merge
                ops.hier_mistakes(self.idx[s], t, counts=self.mistake_counts, node_splits=node_splits,
                                  **self.mistakes.args())
            if self.class_counts is not None and self.row_hi > self.row_lo:
                ops.class_hits(self.idx[s], t, self.class_counts, node_splits=node_splits)
            if self.host_io:
                self.host_counters[s].copy_(self.counters, non_blocking=True)
            return
        if work is not None:
            work.wait()
        pv, pi = unpack_gathered(self.recv[s])
        self.val[s], self.idx[s] = ops.topk_merge(pv, pi, targets=self.dev_labels[s], hits=self.hits)

    def _hier_shard(self) -> Optional[HierShard]:
        return self.hier if self.splits is None else self.splits.hier

    def _issue(self):
        if self.exchange == "p2p":
            return self._issue_p2p()
        prev = None
        for s in range(self.steps):
            work = self._local(s)
            if prev is not None:
                self._merge(*prev)
            prev = (s, work)
        self._merge(*prev)

    def _issue_p2p(self):
        """Fork the current stream into the channel streams, batch s on channel s % channels, join again (inside a
        capture this becomes a graph with `channels` parallel branches)."""
        main = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(main)
        for st in self.side:
            st.wait_event(fork)
        for s in range(self.steps):
            with torch.cuda.stream(self.side[s % self.channels]):
                self._local(s)
                self._merge(s, None)
        for st in self.side:
            join = torch.cuda.Event()
            join.record(st)
            main.wait_event(join)

    def run(self):
        """Score the ``steps`` batches currently in ``dev_feats`` / ``dev_labels`` (enqueue only)."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._issue()

    def close(self) -> None:
        """Release the peer-memory allocations (exchange buffers, peer-visible bank shards).  Call it on every rank,
        after the last replay has finished; the stream must not be used afterwards."""
        torch.cuda.synchronize(self.device)
        self.graph = None
        if self.world > 1:
            dist.barrier(group=self.group)     # nobody unmaps a buffer a peer may still be writing
        for px in getattr(self, "pxs", []):
            px.close()
        for pb in getattr(self, "pbanks", []):
            pb.close()
        self.pxs, self.pbanks = [], []

    def all_reduce_hits(self) -> torch.Tensor:
        """Hit@k counters of the whole batch stream.  With the peer exchange every rank counted its own rows, so
        the counters are summed over ranks (the single collective of an evaluation); the NCCL exchange already
        counts all rows on every rank."""
        h = self.hits.clone()
        if self.exchange == "p2p" and self.world > 1:
            dist.all_reduce(h, group=self.group)
        return h

    # ------------------------------------------------------------------ readout (evaluate.EvalCounters)
    # Every readout is a collective (one all_reduce of the counters): call it on every rank.
    def _read_counters(self, counters):
        torch.cuda.synchronize(self.device)
        if self.world == 1:
            return counters
        c = counters.clone()
        dist.all_reduce(c, group=self.group)
        return c

    def hier_ratios(self):
        """``(hit_ratio, path_ratio, point_ratio)`` in percent -- the TOR / POR of the reference's ``test()`` line -- over
        the rows of all ranks scored so far whose label lies in the hierarchy.  Needs ``hier``."""
        return self.tally.hier_ratios()

    def split_hit_counts(self):
        """Per split ``[Hit@1, @2, @5, @10, @20, rows]`` over the rows of all ranks scored so far, in the order of
        ``splits.names``.  Needs ``splits``."""
        return self.tally.split_hit_counts()

    def split_ratios(self):
        """Per split ``(hit_ratio, path_ratio, point_ratio)`` in percent over the rows of all ranks whose label is in the
        split.  Needs a ``SplitShard`` with ``hier``."""
        return self.tally.split_ratios()

    def split_lines(self):
        """One ``evaluate.split_line`` per split (Hit@k, plus TOR / POR when the ``SplitShard`` has ``hier`` and the
        mistake metrics with ``mistakes`` and the class-averaged Hit@k with ``classes``)."""
        return self.tally.split_lines(self.splits.names)

    def mistake_summary(self):
        """``evaluate.mistake_summary`` over the rows of all ranks scored so far.  Needs ``mistakes`` without
        ``splits``."""
        return self.tally.mistake_summary()

    def split_mistake_summary(self):
        """Per split ``evaluate.mistake_summary`` over the rows of all ranks whose label is in the split.  Needs
        ``mistakes`` and ``splits``."""
        return self.tally.split_mistake_summary()

    def class_table(self) -> torch.Tensor:
        """The per-class table over the rows of all ranks scored so far, host int64 ``[n_nodes, 6]`` (``[S, n_nodes,
        6]`` with ``splits``).  Needs ``classes``."""
        return self.tally.class_table()

    def class_summary(self):
        """``evaluate.class_summary`` over the rows of all ranks scored so far.  Needs ``classes`` without ``splits``."""
        return self.tally.class_summary()

    def split_class_summary(self):
        """Per split ``evaluate.class_summary`` over the rows of all ranks whose label is in the split.  Needs
        ``classes`` and ``splits``."""
        return self.tally.split_class_summary()
