"""Host side of the fused score + mask + top-k call: tensors -> raw pointers -> C ABI.

PyTorch is used for device memory, streams and (in dist.py) torch.distributed only.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import torch

from . import _lib
from ._lib import MASK_ADD, MASK_NONE, MASK_SET  # noqa: F401


def _require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (ccr_b200 has no CPU path)")


def _stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream


class _Workspace:
    """Scratch that only grows, one buffer per (device, stream): calls on different streams (or from
    threads that use different streams) never share candidate / threshold state.  Calls issued on one
    stream are ordered by it, so they may reuse the buffer.  Owned by the caller side of the ABI."""

    def __init__(self):
        self._buf = {}

    def get(self, device, nbytes):
        # never smaller than 256 bytes: a size query that rejected its arguments returns 0, and the call
        # itself, given a valid buffer, then reports why
        nbytes = max(int(nbytes), 256)
        index = device.index if device.index is not None else torch.cuda.current_device()
        key = (device.type, index, torch.cuda.current_stream(device).cuda_stream)
        b = self._buf.get(key)
        if b is None or b.numel() < nbytes:
            b = None
            self._buf[key] = None
            b = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
            # the old block may still be in use by work queued on this stream; the caching allocator
            # only recycles it for the same stream, i.e. after that work
            self._buf[key] = b
        return b

    def clear(self):
        self._buf.clear()


workspace = _Workspace()

_status_record = None


def _status():
    """Host-mapped watchdog record shared with the library (ccr_set_status_record): readable after a
    device trap has poisoned the context."""
    global _status_record
    if _status_record is None:
        _status_record = torch.zeros(4, dtype=torch.int32).pin_memory()
        _lib.lib().ccr_set_status_record(_status_record.data_ptr())
    return _status_record


def device_status():
    """{code, where, block, extra} written by the kernels' bounded barrier waits (code 0 = ok)."""
    c, w, b, x = (int(v) for v in _status())
    return {"code": c, "where": w, "block": b, "extra": x}


def synchronize(device=None):
    """torch.cuda.synchronize that decodes the watchdog record when the device reports a failure."""
    try:
        torch.cuda.synchronize(device)
    except RuntimeError as e:
        st = device_status()
        if st["code"]:
            raise RuntimeError(f"libccr_b200 watchdog: barrier wait timed out (where={st['where']}, "
                               f"block={st['block']}, parity={st['extra']}); CUDA said: {e}") from e
        raise


class SparseMask:
    """Device CSR over item columns: the history / block mask and additive priors.

    ``mode`` MASK_SET: value assigned (ranking(): -1e6, scripts/ms_marco_eval.py:227);
    MASK_ADD: value added in float64 (rime_lite prior_score, src/rime_lite/dataset/base.py:234,279-282).
    Columns are sorted and unique per row (duplicates: summed for ADD, collapsed for SET).
    """

    _f32_exact = None

    def __init__(self, indptr, cols, vals, n_cols, mode, device):
        self.n_rows = len(indptr) - 1
        self.n_cols = int(n_cols)
        self.mode = mode
        self.nnz = int(indptr[-1])
        self.host = (np.asarray(indptr, dtype=np.int64), np.asarray(cols, dtype=np.int32),
                     np.asarray(vals, dtype=np.float64))
        self.max_row_nnz = int(np.diff(self.host[0]).max()) if self.n_rows else 0
        self.device = torch.device(device)
        # pinned staging + non-blocking copies: a pageable upload would make the host wait for all
        # queued device work (per-step mask shards of a row-sharded search are built on the host)
        self.indptr, self.cols, self.vals = (self._upload(a) for a in self.host)

    def _upload(self, a):
        t = torch.as_tensor(a)
        if self.device.type == "cuda" and t.numel():
            return t.pin_memory().to(self.device, non_blocking=True)
        return t.to(self.device)


    @classmethod
    def from_device_tensors(cls, indptr, cols, vals, host, n_cols, mode, nnz=None, max_row_nnz=None,
                            f32_exact=None):
        """Wrap CSR arrays that are already (being copied) on the device; ``host`` holds the same
        arrays as numpy for the host-side slicing helpers, or is None for a CSR that only exists on
        the device -- then ``nnz`` / ``max_row_nnz`` are upper bounds (the C ABI accepts bounds)."""
        self = cls.__new__(cls)
        self.n_rows = int(indptr.shape[0]) - 1
        self.n_cols = int(n_cols)
        self.mode = mode
        self.host = host
        self.nnz = int(host[0][-1]) if nnz is None else int(nnz)
        if max_row_nnz is None:
            max_row_nnz = int(np.diff(host[0]).max()) if self.n_rows else 0
        self.max_row_nnz = int(max_row_nnz)
        self.device = indptr.device
        self.indptr, self.cols, self.vals = indptr, cols, vals
        self._f32_exact = f32_exact
        return self

    @property
    def f32_exact(self):
        """True when ranking by float32 keys is exact for this mask: SET mode with values that are
        float32 numbers (-1e6 is).  ADD priors are summed in float64 and never qualify."""
        if self._f32_exact is None:
            v = self.host[2]
            self._f32_exact = bool(self.mode == MASK_SET and np.array_equal(v.astype(np.float32).astype(np.float64), v))
        return self._f32_exact

    @classmethod
    def from_scipy(cls, csr, mode, device):
        import scipy.sparse as sps

        m = sps.csr_matrix(csr, dtype=np.float64, copy=True)
        if mode == MASK_SET:
            m.data[:] = np.where(m.data == 0, 0.0, m.data)
            # collapse duplicates without summing: keep first
            coo = m.tocoo()
            key = coo.row.astype(np.int64) * m.shape[1] + coo.col
            _, first = np.unique(key, return_index=True)
            m = sps.csr_matrix((coo.data[first], (coo.row[first], coo.col[first])), shape=m.shape)
        else:
            m.sum_duplicates()
        m.sort_indices()
        return cls(m.indptr, m.indices, m.data, m.shape[1], mode, device)

    @classmethod
    def from_lists(cls, rows_of_cols, n_cols, value, mode, device):
        """rows_of_cols: iterable of per-row iterables of column positions (duplicates allowed)."""
        indptr, cols = [0], []
        for r in rows_of_cols:
            u = np.unique(np.asarray(list(r), dtype=np.int64))
            if u.size and (u[0] < 0 or u[-1] >= n_cols):
                raise IndexError("mask column out of range")
            cols.append(u)
            indptr.append(indptr[-1] + u.size)
        cols = np.concatenate(cols) if cols else np.zeros(0, dtype=np.int64)
        vals = np.full(cols.shape, float(value))
        return cls(indptr, cols, vals, n_cols, mode, device)

    @classmethod
    def from_flat(cls, row_lengths, cols, n_cols, value, mode, device):
        """Rows given back to back: ``cols`` holds row 0's columns, then row 1's, ... (duplicates
        allowed); ``row_lengths[r]`` entries belong to row r.  One vectorised sort instead of a
        Python loop over rows (block lists of whole brands: ~1.3 M entries for 9,862 queries)."""
        row_lengths = np.asarray(row_lengths, dtype=np.int64)
        cols = np.asarray(cols, dtype=np.int64)
        if cols.size and (cols.min() < 0 or cols.max() >= n_cols):
            raise IndexError("mask column out of range")
        row_of = np.repeat(np.arange(len(row_lengths), dtype=np.int64), row_lengths)
        key = np.sort(row_of * np.int64(n_cols) + cols)     # by (row, col); sort + diff: np.unique is 50x slower
        if key.size:
            key = key[np.concatenate(([True], key[1:] != key[:-1]))]
        rows_u, cols_u = key // n_cols, key % n_cols
        indptr = np.zeros(len(row_lengths) + 1, dtype=np.int64)
        np.cumsum(np.bincount(rows_u, minlength=len(row_lengths)), out=indptr[1:])
        return cls(indptr, cols_u, np.full(cols_u.shape, float(value)), n_cols, mode, device)

    def rows(self, start, stop):
        ip, c, v = self.host
        a, b = ip[start], ip[stop]
        return SparseMask(ip[start : stop + 1] - a, c[a:b], v[a:b], self.n_cols, self.mode, self.device)

    def take_rows(self, rows):
        """The CSR of the given rows (host int array), in that order."""
        if self.host is None:
            raise NotImplementedError("take_rows needs the host copy of the CSR")
        ip, c, v = self.host
        rows = np.asarray(rows, dtype=np.int64)
        lengths = ip[rows + 1] - ip[rows]
        new_ip = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        src = np.repeat(ip[rows] - new_ip[:-1], lengths) + np.arange(new_ip[-1], dtype=np.int64)
        return SparseMask(new_ip, c[src], v[src], self.n_cols, self.mode, self.device)

    def column_shard_device(self, lo, hi):
        """column_shard on the device (C ABI: ccr_mask_column_shard): no host pass, no upload.  The
        shard's entry count stays on the device; nnz / max_row_nnz of the result are upper bounds."""
        _require_cuda(self.indptr, "mask")
        dev = self.indptr.device
        out_ip = torch.empty_like(self.indptr)
        out_c = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
        out_v = torch.empty(max(self.nnz, 1), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = _lib.lib().ccr_mask_column_shard(self.indptr.data_ptr(), self.cols.data_ptr() if self.nnz else None,
                                                  self.vals.data_ptr() if self.nnz else None, self.n_rows, int(lo), int(hi),
                                                  out_ip.data_ptr(), out_c.data_ptr(), out_v.data_ptr(), _stream_ptr(dev))
        _lib.check(rc)
        return SparseMask.from_device_tensors(out_ip, out_c, out_v, None, hi - lo, self.mode, nnz=self.nnz,
                                              max_row_nnz=self.max_row_nnz, f32_exact=self.f32_exact)

    def column_shard(self, lo, hi):
        """Entries with lo <= col < hi, re-based to local column ids (row-sharded tables)."""
        ip, c, v = self.host
        keep = (c >= lo) & (c < hi)
        row_of = np.repeat(np.arange(self.n_rows), np.diff(ip))
        counts = np.bincount(row_of[keep], minlength=self.n_rows)
        new_ip = np.concatenate([[0], np.cumsum(counts)])
        return SparseMask(new_ip, c[keep] - lo, v[keep], hi - lo, self.mode, self.device)


_MaskABI = namedtuple("_MaskABI", "indptr cols vals nnz h_max mode")
_NO_MASK = _MaskABI(None, None, None, 0, -1, MASK_NONE)


def _mask_abi(mask, B, N):
    """The C ABI arguments of ``mask`` for B rows and N columns: raw pointers, nnz, max row nnz and mode, or
    None when there is no mask to apply (None, MASK_NONE or no entries): the rule the C ABI applies, so every
    wrapper passes the same arguments for the same mask."""
    if mask is None:
        return None
    if mask.n_rows != B or mask.n_cols != N:
        raise ValueError(f"mask shape ({mask.n_rows}, {mask.n_cols}) does not match ({B}, {N})")
    if mask.mode == MASK_NONE or mask.nnz <= 0:
        return None
    return _MaskABI(mask.indptr.data_ptr(), mask.cols.data_ptr(), mask.vals.data_ptr(), mask.nnz, mask.max_row_nnz,
                    mask.mode)


def _rows_pitch(t):
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def _operand_f16(q, items):
    """True for two fp16 operands, False for two bf16 ones; anything else is a TypeError."""
    if q.dtype == items.dtype == torch.float16:
        return True
    if q.dtype == items.dtype == torch.bfloat16:
        return False
    if {q.dtype, items.dtype} <= {torch.bfloat16, torch.float16}:
        raise TypeError(f"q is {q.dtype} but items are {items.dtype}: encode the queries with the table "
                        "(EmbeddingTable.encode_queries) so both share its dtype")
    raise TypeError("q and items must both be bfloat16 or both float16 (use EmbeddingTable / ingest_rows to convert)")


def score_topk(q, items, k, mask: SparseMask | None = None, id_offset=0, algo=_lib.ALGO_AUTO,
               allow_short=False, want_f64=False, n_items=None, D=None, want_keys=False):
    """Fused ``topk(q @ items.T [mask], k)`` on the device (C ABI: ccr_score_topk_bf16).

    q [B, ldq] bf16 cuda, items [N, ldi] bf16 cuda (row-major, last dim contiguous); or both fp16
    (CCR_FLAG_F16: fp16 operands, fp32 accumulation, fp32 scores).
    Returns (scores float32 [B,k] descending, ids int64 [B,k]) and, with ``want_f64``, the
    float64 values the order was decided on; with ``want_keys`` instead the packed uint64
    exchange keys (CCR_FLAG_PACKED_KEYS; int64 tensor holding the bit pattern).
    """
    _require_cuda(q, "q")
    _require_cuda(items, "items")
    f16 = _operand_f16(q, items)
    if q.dim() != 2 or items.dim() != 2 or q.stride(1) != 1 or items.stride(1) != 1:
        raise ValueError("q and items must be 2-d with a contiguous last dimension")
    dev = q.device
    B = q.shape[0]
    N = items.shape[0] if n_items is None else int(n_items)
    D = q.shape[1] if D is None else int(D)
    ldq, ldi = _rows_pitch(q), _rows_pitch(items)
    k = int(k)
    flags = int(algo) | (_lib.FLAG_ALLOW_SHORT if allow_short else 0) | (_lib.FLAG_F16 if f16 else 0)
    if want_keys:
        if want_f64:
            raise ValueError("want_keys and want_f64 are exclusive (one 8-byte slot per entry)")
        flags |= _lib.FLAG_PACKED_KEYS
    L = _lib.lib()
    m = _mask_abi(mask, B, N) or _NO_MASK
    out_s = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
    out_d = torch.empty((B, k), dtype=torch.float64, device=dev) if want_f64 else None
    if want_keys:
        out_d = torch.empty((B, k), dtype=torch.int64, device=dev)
    _status()
    with torch.cuda.device(dev):
        ws = workspace.get(dev, L.ccr_score_topk_workspace_bytes(B, N, D, k, m.nnz, m.h_max, flags))
        rc = L.ccr_score_topk_bf16(
            q.data_ptr(), B, ldq, items.data_ptr() if N > 0 else None, N, ldi, D, k,
            m.indptr, m.cols, m.vals, m.nnz, m.h_max, m.mode, int(id_offset),
            out_s.data_ptr(), out_d.data_ptr() if out_d is not None else None, out_i.data_ptr(),
            ws.data_ptr(), ws.numel(), flags, _stream_ptr(dev))
    _lib.check(rc)
    return (out_s, out_i, out_d) if out_d is not None else (out_s, out_i)


def merge_topk(scores64, ids, k_out):
    """[G,B,k_in] float64 / int64 sorted runs -> merged top-k_out (C ABI: ccr_merge_topk)."""
    _require_cuda(scores64, "scores64")
    G, B, k_in = scores64.shape
    scores64 = scores64.contiguous()
    ids = ids.contiguous()
    dev = scores64.device
    out_s = torch.empty((B, k_out), dtype=torch.float32, device=dev)
    out_d = torch.empty((B, k_out), dtype=torch.float64, device=dev)
    out_i = torch.empty((B, k_out), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib().ccr_merge_topk(scores64.data_ptr(), ids.data_ptr(), G, B, k_in, k_out, out_s.data_ptr(),
                                       out_d.data_ptr(), out_i.data_ptr(), _stream_ptr(dev))
    _lib.check(rc)
    return out_s, out_i, out_d


def merge_topk_keys(keys, k_out, packed=False):
    """[G,B,k_in] packed exchange keys (int64 bit patterns) -> merged (scores f32, ids i64) [B,k_out], or
    with ``packed`` the merged runs still as keys [B,k_out] (C ABI: ccr_merge_topk_keys)."""
    _require_cuda(keys, "keys")
    G, B, k_in = keys.shape
    keys = keys.contiguous()
    dev = keys.device
    if packed:
        out_k = torch.empty((B, k_out), dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            rc = _lib.lib().ccr_merge_topk_keys(keys.data_ptr(), G, B, k_in, k_out, None, None, out_k.data_ptr(),
                                                _stream_ptr(dev))
        _lib.check(rc)
        return out_k
    out_s = torch.empty((B, k_out), dtype=torch.float32, device=dev)
    out_i = torch.empty((B, k_out), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib().ccr_merge_topk_keys(keys.data_ptr(), G, B, k_in, k_out, out_s.data_ptr(), out_i.data_ptr(), None,
                                            _stream_ptr(dev))
    _lib.check(rc)
    return out_s, out_i


def unpack_topk_keys(keys):
    """Packed exchange keys (any shape, int64 bit patterns) -> (scores f32, ids i64) of the same shape
    (C ABI: ccr_unpack_topk_keys)."""
    _require_cuda(keys, "keys")
    keys = keys.contiguous()
    dev = keys.device
    out_s = torch.empty(keys.shape, dtype=torch.float32, device=dev)
    out_i = torch.empty(keys.shape, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib().ccr_unpack_topk_keys(keys.data_ptr(), keys.numel(), out_s.data_ptr(), out_i.data_ptr(),
                                             _stream_ptr(dev))
    _lib.check(rc)
    return out_s, out_i


def topk_dense(scores, k, mask: SparseMask | None = None):
    """Top-k of a materialised float32 score matrix [B, N] on the device (+ sparse prior, float64
    like the reference's promotion): C ABI ccr_topk_dense_f32.  Returns (scores f32, ids i64, scores f64)."""
    _require_cuda(scores, "scores")
    if scores.dtype != torch.float32 or scores.dim() != 2 or (scores.shape[1] and scores.stride(1) != 1):
        raise TypeError("scores must be a 2-d float32 tensor with a contiguous last dimension")
    B, N = scores.shape
    k = int(k)
    dev = scores.device
    m = _mask_abi(mask, B, N) or _NO_MASK
    out_s = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_d = torch.empty((B, k), dtype=torch.float64, device=dev)
    out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        ws = workspace.get(dev, L.ccr_topk_dense_workspace_bytes(B, N, k, m.nnz, m.h_max))
        rc = L.ccr_topk_dense_f32(
            scores.data_ptr(), B, N, _rows_pitch(scores), k, m.indptr, m.cols, m.vals, m.nnz, m.h_max, m.mode,
            out_s.data_ptr(), out_d.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(dev))
    _lib.check(rc)
    return out_s, out_i, out_d


def argsort_scores(scores, mask: SparseMask | None = None):
    """Whole-matrix argsort of a float32 score matrix [B, N] on the device (+ sparse prior in float64),
    best first, equal scores in flat order: (rows int64 [B*N], cols int64 [B*N]).  C ABI:
    ccr_argsort_scores_f32 (LSD radix sort)."""
    _require_cuda(scores, "scores")
    if scores.dtype != torch.float32 or scores.dim() != 2 or (scores.shape[1] and scores.stride(1) != 1):
        raise TypeError("scores must be a 2-d float32 tensor with a contiguous last dimension")
    B, N = scores.shape
    dev = scores.device
    n = B * N
    m = _mask_abi(mask, B, N) or _NO_MASK
    rows = torch.empty(n, dtype=torch.int64, device=dev)
    cols = torch.empty(n, dtype=torch.int64, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        need = L.ccr_argsort_workspace_bytes(n)
        if need == 0 and n > 0:
            raise ValueError("argsort: more than 2^31 matrix elements")
        ws = workspace.get(dev, need)
        rc = L.ccr_argsort_scores_f32(scores.data_ptr(), B, N, _rows_pitch(scores), m.indptr, m.cols, m.vals, m.nnz,
                                      m.mode, rows.data_ptr(), cols.data_ptr(), ws.data_ptr(), ws.numel(),
                                      _stream_ptr(dev))
    _lib.check(rc)
    return rows, cols


def first_hit_rank(ids, rel_indptr, rel_ids):
    """Per row of ``ids`` [B, k] (ranked, int64, device) the 1-based rank of the first id found in the
    row's sorted relevant list (CSR: rel_indptr int64 [B+1], rel_ids int64), 0 = none.  C ABI:
    ccr_first_hit_rank.  Returns int32 [B] on the device."""
    _require_cuda(ids, "ids")
    if ids.dtype != torch.int64 or ids.dim() != 2:
        raise TypeError("ids must be a 2-d int64 tensor")
    ids = ids.contiguous()
    B, k = ids.shape
    dev = ids.device
    rel_indptr = torch.as_tensor(rel_indptr, dtype=torch.int64).to(dev)
    rel_ids = torch.as_tensor(rel_ids, dtype=torch.int64).to(dev)
    if rel_indptr.numel() != B + 1:
        raise ValueError("rel_indptr must have B + 1 entries")
    out = torch.empty(B, dtype=torch.int32, device=dev)
    if B == 0:
        return out
    with torch.cuda.device(dev):
        rc = _lib.lib().ccr_first_hit_rank(ids.data_ptr(), B, k, rel_indptr.data_ptr(),
                                           rel_ids.data_ptr() if rel_ids.numel() else None, out.data_ptr(),
                                           _stream_ptr(dev))
    _lib.check(rc)
    return out


def ingest_rows(src, dst, normalize=False, overflow=None):
    """fp32 (or bf16 / fp16) rows on the device -> bf16 or fp16 table rows (``dst.dtype``), optional fp32
    L2 normalisation.  fp16 destinations: ``overflow`` (a device int32 [1] tensor, optional) has the
    number of stored values that are not finite added to it (|x| >= 65520 rounds to inf)."""
    _require_cuda(src, "src")
    _require_cuda(dst, "dst")
    if dst.dtype not in (torch.bfloat16, torch.float16) or dst.stride(1) != 1 or src.stride(1) != 1:
        raise ValueError("dst must be bf16 or fp16 and both must have a contiguous last dimension")
    n, D = src.shape
    if dst.shape[0] != n or dst.shape[1] < D:
        raise ValueError("dst shape mismatch")
    if n > 1 and dst.stride(0) != dst.shape[1]:
        # the kernel zero-fills every column up to the row pitch: a column slice of a wider tensor
        # would have its neighbours overwritten
        raise ValueError("dst rows must be dense (stride(0) == shape[1])")
    f16 = dst.dtype == torch.float16
    if f16 and src.dtype == torch.bfloat16:
        src = src.float()  # bf16 -> fp32 is exact; the fp16 rounding happens once, in the kernel
    if not f16 and src.dtype == torch.float16:
        raise TypeError("fp16 rows do not go into a bf16 table: pass them as float32")
    if overflow is not None and (not f16 or overflow.dtype != torch.int32 or not overflow.is_cuda):
        raise ValueError("overflow must be a device int32 tensor, for fp16 destinations only")
    ld_src, ld_dst = _rows_pitch(src), _rows_pitch(dst)
    L = _lib.lib()
    with torch.cuda.device(src.device):
        if src.dtype == torch.float32:
            if f16:
                rc = L.ccr_ingest_rows_f32_f16(src.data_ptr(), n, D, ld_src, dst.data_ptr(), ld_dst,
                                               int(bool(normalize)),
                                               overflow.data_ptr() if overflow is not None else None,
                                               _stream_ptr(src.device))
            else:
                rc = L.ccr_ingest_rows_f32(src.data_ptr(), n, D, ld_src, dst.data_ptr(), ld_dst, int(bool(normalize)),
                                           _stream_ptr(src.device))
        elif src.dtype == dst.dtype:
            if not normalize:
                dst[:, :D].copy_(src)
                if dst.shape[1] > D:
                    dst[:, D:].zero_()
                return dst
            fn = L.ccr_normalize_rows_f16 if f16 else L.ccr_normalize_rows_bf16
            rc = fn(src.data_ptr(), n, D, ld_src, dst.data_ptr(), ld_dst, _stream_ptr(src.device))
        else:
            raise TypeError(f"unsupported source dtype {src.dtype}")
    _lib.check(rc)
    return dst


def score_dense(q, items, n_items=None, D=None):
    """Dense fp32 [B, N] scores (small reranking sets / LazyScore.as_tensor); bf16 or fp16 operands."""
    _require_cuda(q, "q")
    f16 = _operand_f16(q, items)
    B = q.shape[0]
    N = items.shape[0] if n_items is None else n_items
    D = q.shape[1] if D is None else D
    out = torch.empty((B, N), dtype=torch.float32, device=q.device)
    if B == 0 or N == 0:
        return out
    with torch.cuda.device(q.device):
        fn = _lib.lib().ccr_score_dense_f16 if f16 else _lib.lib().ccr_score_dense_f32
        rc = fn(q.data_ptr(), B, _rows_pitch(q), items.data_ptr(), N, _rows_pitch(items), D, out.data_ptr(), N,
                _stream_ptr(q.device))
    _lib.check(rc)
    return out


# ---- exact fp32 ranking (DESIGN.md section 6b) ----

def exact_error_bound(q_norm, v_max, D, f16):
    """Python mirror of ``exact_error_bound`` (csrc/ccr_common.cuh, exported as ccr_exact_error_bound): a
    bound of |scan score - exact value| for a query of norm ``q_norm`` against a table whose largest fp32
    row norm is ``v_max``.  Works elementwise on numpy arrays."""
    u = 2.0 ** -11 if f16 else 2.0 ** -8
    eta = 2.0 ** -25 if f16 else 2.0 ** -134
    d = float(D)
    qv = np.asarray(q_norm, dtype=np.float64) * v_max
    under = (1.0 + u) * eta * np.sqrt(d) * (np.asarray(q_norm, dtype=np.float64) + v_max) + d * eta * eta
    a = (1.0 + u) * (1.0 + u) * qv + under
    e = (2.0 * u + u * u) * qv + under + d * 2.0 ** -22 * a + d * 2.0 ** -149 + (2.0 ** -24 + d * 2.0 ** -53) * qv
    return e * (1.0 + 2.0 ** -20)


# scan-score rows of the fallback are computed in blocks of at most this many bytes: every block streams the
# whole scan table once, so larger blocks mean fewer passes (4 GB: ~120 rows per pass at 8.84 M items)
EXACT_FALLBACK_BLOCK_BYTES = 4 << 30


def ingest_rows_f32(src, dst, normalize=False, v_max=None):
    """fp32 rows -> fp32 rows of an exact table (optional fp32 L2 normalisation, zeroed padding columns);
    ``v_max`` (device float64 [1], optional) is raised to the largest stored row norm (rounded up)."""
    _require_cuda(src, "src")
    _require_cuda(dst, "dst")
    if src.dtype != torch.float32 or dst.dtype != torch.float32 or src.stride(1) != 1 or dst.stride(1) != 1:
        raise ValueError("src and dst must be float32 with a contiguous last dimension")
    n, D = src.shape
    if dst.shape[0] != n or dst.shape[1] < D or (n > 1 and dst.stride(0) != dst.shape[1]):
        raise ValueError("dst must be dense rows [n, >= D]")
    if v_max is not None and (v_max.dtype != torch.float64 or not v_max.is_cuda):
        raise ValueError("v_max must be a device float64 tensor")
    with torch.cuda.device(src.device):
        rc = _lib.lib().ccr_ingest_rows_f32_f32(src.data_ptr(), n, D, _rows_pitch(src), dst.data_ptr(),
                                                _rows_pitch(dst), int(bool(normalize)),
                                                v_max.data_ptr() if v_max is not None else None,
                                                _stream_ptr(src.device))
    _lib.check(rc)
    return dst


def score_topk_exact(q, q_scan, items, items_scan, k, v_max, mask: SparseMask | None = None, id_offset=0,
                     algo=_lib.ALGO_AUTO, allow_short=False, n_items=None, D=None):
    """Exact fp32 top-k (C ABI: ccr_score_topk_exact, then the fallback for uncertified rows).

    q [B, ld] / items [N, ld] fp32 rows, q_scan / items_scan their bf16 or fp16 rounding (same pitch),
    v_max the device float64 [1] largest fp32 row norm of items.  Returns (scores float32, ids int64,
    values float64, number of rows that went through the fallback)."""
    for t, name in ((q, "q"), (items, "items"), (q_scan, "q_scan"), (items_scan, "items_scan")):
        _require_cuda(t, name)
    f16 = _operand_f16(q_scan, items_scan)
    if q.dtype != torch.float32 or items.dtype != torch.float32:
        raise TypeError("q and items must be the float32 rows of an exact table")
    if q.stride() != q_scan.stride() or items.stride() != items_scan.stride():
        raise ValueError("the fp32 rows and their scan copies must share one row pitch")
    dev = q.device
    B = q.shape[0]
    N = items.shape[0] if n_items is None else int(n_items)
    D = q.shape[1] if D is None else int(D)
    k = int(k)
    ldq, ldi = _rows_pitch(q), _rows_pitch(items)
    flags = int(algo) | (_lib.FLAG_ALLOW_SHORT if allow_short else 0) | (_lib.FLAG_F16 if f16 else 0)
    m = _mask_abi(mask, B, N) or _NO_MASK
    out_s = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
    out_d = torch.empty((B, k), dtype=torch.float64, device=dev)
    uncert = torch.empty(B, dtype=torch.int32, device=dev)
    tau = torch.empty(B, dtype=torch.float64, device=dev)
    count = torch.zeros(1, dtype=torch.int32, device=dev)
    L = _lib.lib()
    _status()
    with torch.cuda.device(dev):
        ws = workspace.get(dev, L.ccr_score_topk_exact_workspace_bytes(B, N, D, k, m.nnz, m.h_max, flags))
        rc = L.ccr_score_topk_exact(
            q.data_ptr(), q_scan.data_ptr(), B, ldq, items.data_ptr() if N else None,
            items_scan.data_ptr() if N else None, N, ldi, D, k, v_max.data_ptr(),
            m.indptr, m.cols, m.vals, m.nnz, m.h_max, m.mode, int(id_offset), out_s.data_ptr(), out_d.data_ptr(),
            out_i.data_ptr(), uncert.data_ptr(), tau.data_ptr(), count.data_ptr(), ws.data_ptr(), ws.numel(), flags,
            _stream_ptr(dev))
    _lib.check(rc)
    n_fallback = int(count.item()) if B else 0
    if n_fallback:
        rows = torch.nonzero(uncert, as_tuple=True)[0]
        block = max(1, min(65535, EXACT_FALLBACK_BLOCK_BYTES // (4 * max(N, 1))))
        for r0 in range(0, rows.numel(), block):
            r = rows[r0 : r0 + block]
            s_r, i_r, d_r = _exact_fallback_rows(q[r], q_scan[r], items, items_scan, k, tau[r], mask, r, id_offset,
                                                 allow_short, N, D)
            out_s[r], out_i[r], out_d[r] = s_r, i_r, d_r
    return out_s, out_i, out_d, n_fallback


def _exact_fallback_rows(q, q_scan, items, items_scan, k, tau, mask, rows, id_offset, allow_short, N, D):
    """The complete path of uncertified rows: dense scan scores, the columns at or above each row's tau,
    exact re-rank of those and the row's mask entries."""
    dev = q.device
    R = q.shape[0]
    L = _lib.lib()
    scores = score_dense(q_scan, items_scan, n_items=N, D=D)
    indptr = torch.empty(R + 1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.ccr_threshold_compact(scores.data_ptr(), R, N, N, tau.data_ptr(), indptr.data_ptr(), None,
                                           _stream_ptr(dev)))
        total = int(indptr[-1].item())
        ids = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        _lib.check(L.ccr_threshold_compact(scores.data_ptr(), R, N, N, tau.data_ptr(), indptr.data_ptr(),
                                           ids.data_ptr(), _stream_ptr(dev)))
    del scores
    m = _mask_abi(mask.take_rows(rows.cpu().numpy()) if mask is not None else None, R, N) or _NO_MASK
    out_s = torch.empty((R, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((R, k), dtype=torch.int64, device=dev)
    out_d = torch.empty((R, k), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        ws = workspace.get(dev, L.ccr_rerank_exact_workspace_bytes(R, total, m.nnz))
        rc = L.ccr_rerank_exact(
            q.data_ptr(), R, _rows_pitch(q), items.data_ptr() if N else None, N, _rows_pitch(items), D, k,
            indptr.data_ptr(), ids.data_ptr(), total, m.indptr, m.cols, m.vals, m.nnz, m.mode, int(id_offset),
            out_s.data_ptr(), out_d.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(),
            _lib.FLAG_ALLOW_SHORT if allow_short else 0, _stream_ptr(dev))
    _lib.check(rc)
    return out_s, out_i, out_d
