"""Row-sharded item table across the GPUs of one box: one process per GPU, local fused
top-k with global ids, then the exchange: packed 8-byte (float32 score, uint32 id) keys go through an
all-to-all (every rank receives all runs of its B/G query rows), an on-device G-way merge-path merge
and an all-gather of the merged rows -- or, when float64 priors decide the order, one all-gather of
(float64 score, int64 id) pairs and the merge of all rows on every rank.  The reference has no counterpart (it scores on GPU 0 only, scripts/ms_marco_eval.py:205).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import engine
from .table import EmbeddingTable, check_table_dtype


def shard_bounds(n_items, world_size, rank):
    """Contiguous row shard [lo, hi) of rank: ceil(N/G) rows each, last shard shorter/empty."""
    per = (n_items + world_size - 1) // world_size
    lo = min(n_items, rank * per)
    hi = min(n_items, lo + per)
    return lo, hi


class ShardedIndex:
    """Each rank holds rows [lo, hi) of the global table in an EmbeddingTable with id_offset=lo."""

    def __init__(self, n_items, dim=768, normalize=False, device=None, group=None, dtype=torch.bfloat16,
                 exact=False):
        self.dtype = check_table_dtype(dtype)  # element type of the local table (bf16 or fp16)
        # exact: local exact top-k (DESIGN.md section 6b), then the (float64, int64) pair exchange; an item's
        # exact value does not depend on the shard that holds it, so the merge equals one exact table
        self.exact = bool(exact)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_items = int(n_items)
        self.lo, self.hi = shard_bounds(self.n_items, self.world, self.rank)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.table = self._make_table(self.hi - self.lo, dim, normalize)

    def _make_table(self, capacity, dim, normalize):
        return EmbeddingTable(capacity, dim, device=self.device, normalize=normalize, id_offset=self.lo,
                              dtype=self.dtype, exact=self.exact)

    # ---- the device steps; CPU gloo tests replace them to exercise the plumbing ----
    def _local_topk(self, q_encoded, k, mask):
        s, i, d = self.table.search(q_encoded, k, mask=mask, allow_short=True, want_f64=True, encoded=True)
        return d, i

    def _local_topk_keys(self, q_encoded, k, mask):
        s, i, keys = self.table.search(q_encoded, k, mask=mask, allow_short=True, want_keys=True, encoded=True)
        return keys

    def _merge(self, scores64, ids, k):
        return engine.merge_topk(scores64, ids, k)

    def _merge_keys(self, keys, k, packed=False):
        return engine.merge_topk_keys(keys, k, packed=packed)

    def _unpack_keys(self, keys):
        return engine.unpack_topk_keys(keys)

    def _exchange_keys(self, keys, k):
        """Local sorted runs [B, k] of packed keys on every rank -> global top-k (scores, ids) on every
        rank.  Query-sharded: an all-to-all hands rank r every rank's runs of ITS slice of the queries
        (B/G rows), it merges only those, and an all-gather of the merged, still packed rows completes
        the result: 2 B k 8 bytes cross each link per rank instead of G B k 8, and every rank merges
        B/G rows instead of B."""
        G, B = self.world, keys.shape[0]
        per = (B + G - 1) // G
        if per * G != B:
            keys = torch.cat([keys, keys.new_zeros((per * G - B, k))])  # key 0 = padding
        recv = torch.empty_like(keys)                       # [G, per, k]: block g = rank g's runs of my rows
        dist.all_to_all_single(recv, keys.contiguous(), group=self.group)
        mine = self._merge_keys(recv.view(G, per, k), k, packed=True)
        full = torch.empty((G * per, k), dtype=keys.dtype, device=keys.device)
        dist.all_gather_into_tensor(full, mine.contiguous(), group=self.group)
        return self._unpack_keys(full[:B])

    def _encode(self, queries):
        return self.table.encode_queries(queries)

    def _shard_mask(self, mask):
        """The rank's column range of the GLOBAL mask, re-based to local columns: on the device when
        the CSR already lives there (no host pass, no upload), else from the host arrays."""
        if mask is None:
            return None
        if getattr(mask, "indptr", None) is not None and mask.indptr.is_cuda and not (self.exact and mask.host is not None):
            # (an exact search's fallback selects mask rows on the host, so it keeps the host copy)
            return mask.column_shard_device(self.lo, self.hi)
        return mask.column_shard(self.lo, self.hi)

    def _encode_replicated(self, queries):
        """Encoded queries (the table's dtype) on every rank.  Host queries are uploaded and encoded in G row
        slices, one per rank, and all-gathered over NVLink: B*D*4/G bytes cross each PCIe link instead of B*D*4."""
        if self.world == 1 or not isinstance(queries, torch.Tensor) or queries.is_cuda or queries.dim() != 2:
            return self._encode(queries)
        B = queries.shape[0]
        per = (B + self.world - 1) // self.world
        a, b = min(B, self.rank * per), min(B, (self.rank + 1) * per)
        part = self._encode(queries[a:b]) if b > a else None
        ld = part.shape[1] if part is not None else self._encode(queries[:1]).shape[1]
        enc_dtype = torch.float32 if self.exact else self.dtype  # exact tables encode queries as fp32 rows
        mine = torch.zeros((per, ld), dtype=enc_dtype if part is None else part.dtype,
                           device=self.device if part is None else part.device)
        if part is not None:
            mine[: b - a].copy_(part)
        full = torch.empty((self.world * per, ld), dtype=mine.dtype, device=mine.device)
        dist.all_gather_into_tensor(full, mine, group=self.group)
        return full[:B]

    def add_local(self, emb):
        """Append rows of this rank's shard (in global order)."""
        self.table.append(emb)
        return self

    def can_pack(self, mask):
        """One all-gather of packed 8-byte (float32 score, uint32 id) keys is exact when the order is
        decided in float32: no mask, or SET values that are float32 numbers; ADD priors (float64
        sums) take the (float64, int64) pair exchange."""
        return not self.exact and self.n_items <= (1 << 32) and (mask is None or mask.f32_exact)

    def search(self, queries, k, mask: engine.SparseMask | None = None, want_f64=False):
        """queries replicated on every rank; mask is the GLOBAL CSR (sharded here by column range).
        Returns (scores f32 [B,k], global ids [B,k], scores f64 [B,k] or None) on every rank; the
        float64 values are only produced on the pair-exchange path (ADD priors or ``want_f64``)."""
        if k > self.n_items:
            raise RuntimeError("selected index k out of range")
        q = self._encode_replicated(queries)
        local_mask = self._shard_mask(mask)
        if self.can_pack(mask) and not want_f64:
            keys = self._local_topk_keys(q, k, local_mask)
            if self.world == 1:
                return (*self._merge_keys(keys.unsqueeze(0), k), None)
            return (*self._exchange_keys(keys, k), None)
        d, i = self._local_topk(q, k, local_mask)
        if self.world == 1:
            return self._merge(d.unsqueeze(0), i.unsqueeze(0), k)
        B = d.shape[0]
        gs = torch.empty((self.world * B, k), dtype=d.dtype, device=d.device)   # rank-major concatenation
        gi = torch.empty((self.world * B, k), dtype=i.dtype, device=i.device)
        dist.all_gather_into_tensor(gs, d.contiguous(), group=self.group)
        dist.all_gather_into_tensor(gi, i.contiguous(), group=self.group)
        return self._merge(gs.view(self.world, B, k), gi.view(self.world, B, k), k)
