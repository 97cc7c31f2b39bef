"""Embedding-table residency layer: a device-resident bf16 (or, opt-in, fp16) [N, ld] item/passage table.

Replaces the reference's pageable host fp32 table (scripts/ms_marco_eval.py:123-152
``generate_embeddings`` -> ``.to("cpu")`` -> ``vstack``; src/ccrec/models/bbpr.py:466-483
``get_all_embeddings``): encoder batches are cast (and, for CCREC_SIM_TYPE=cos, L2-normalised
in fp32) straight into the device table, which then never crosses PCIe again.
"""
from __future__ import annotations

import torch

from . import engine


def _round_up(x, m):
    return (x + m - 1) // m * m


TABLE_DTYPES = (torch.bfloat16, torch.float16)
_DTYPE_NAMES = {torch.bfloat16: "bfloat16", torch.float16: "float16"}


def check_table_dtype(dtype):
    """The element type of a device table: bf16 (default) or fp16; anything else is a ValueError."""
    if dtype not in TABLE_DTYPES:
        raise ValueError(f"table dtype must be torch.bfloat16 or torch.float16, not {dtype}")
    return dtype


class EmbeddingTable:
    """Row-major bf16 table on one GPU.  ``id_offset`` is the global id of local row 0
    (row-sharded tables: scripts-level corpus position = id_offset + local row).

    ``dtype=torch.float16`` stores IEEE fp16 instead: the operand format of the reference's autocast GPU
    matmul (scripts/al_0_rank.py:125), 11 significant bits instead of 8, same 2 bytes per element and
    the same kernels (fp32 accumulation, fp32 scores).  fp16 overflows above 65504: an append or a
    query batch with a value that rounds to inf is refused with ValueError.

    ``exact=True`` keeps the fp32 rows as well (6 bytes per element) and ``search`` returns the exact fp32
    ranking (DESIGN.md section 6b): ``dtype`` is then the format of the scan copy that the fused kernel
    reads, and the candidates it returns are re-scored from the fp32 rows with a certificate that no other
    item can reach the top k (fp16 scans need far fewer candidates than bf16 ones)."""

    def __init__(self, capacity, dim=768, device="cuda", normalize=False, id_offset=0, dtype=torch.bfloat16,
                 exact=False):
        self.dtype = check_table_dtype(dtype)
        self.dim = int(dim)
        self.ld = _round_up(self.dim, 8)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("EmbeddingTable lives on a CUDA device (ccr_b200 has no CPU path)")
        self.normalize = bool(normalize)
        self.id_offset = int(id_offset)
        self.data = torch.empty((int(capacity), self.ld), dtype=self.dtype, device=self.device)
        self.exact = bool(exact)
        # exact tables: the fp32 rows and their largest norm (V of the error bound, device float64 [1])
        self.data32 = torch.empty((int(capacity), self.ld), dtype=torch.float32, device=self.device) if exact else None
        self.v_max = torch.zeros(1, dtype=torch.float64, device=self.device) if exact else None
        self.n = 0

    def __len__(self):
        return self.n

    @property
    def rows(self):
        return self.data[: self.n]

    def nbytes(self):
        return self.n * self.ld * (6 if self.exact else 2)

    def append(self, emb):
        """Append a batch of embeddings [m, dim] (any device / float dtype)."""
        emb = torch.as_tensor(emb)
        if emb.dim() == 1:
            emb = emb.unsqueeze(0)
        m = emb.shape[0]
        if emb.shape[1] != self.dim:
            raise ValueError(f"embedding dim {emb.shape[1]} != table dim {self.dim}")
        if self.n + m > self.data.shape[0]:
            grown = torch.empty((max(self.n + m, 2 * self.data.shape[0]), self.ld), dtype=self.dtype,
                                device=self.device)
            grown[: self.n].copy_(self.data[: self.n])
            self.data = grown
            if self.exact:
                grown = torch.empty((self.data.shape[0], self.ld), dtype=torch.float32, device=self.device)
                grown[: self.n].copy_(self.data32[: self.n])
                self.data32 = grown
        if self.exact:
            v = torch.zeros(1, dtype=torch.float64, device=self.device)
            self._ingest_exact(emb, self.data32[self.n : self.n + m], self.data[self.n : self.n + m], v)
            torch.maximum(self.v_max, v, out=self.v_max)  # only once the batch was accepted
        else:
            self._ingest(emb, self.data[self.n : self.n + m])
        self.n += m
        return self

    def _ingest(self, src, dst, normalize=None):
        """Rows of any float dtype -> ``dst`` under the table's dtype and similarity convention (``normalize``
        overrides the table's).  fp32 and table-dtype sources go to the kernels as they are; everything else
        is widened to fp32 first."""
        normalize = self.normalize if normalize is None else normalize
        if src.dtype not in (torch.float32, self.dtype):
            src = src.float()
        src = src.to(self.device, non_blocking=True)
        if src.stride(1) != 1:
            src = src.contiguous()
        if self.dtype == torch.bfloat16 or src.dtype != torch.float32:
            return engine.ingest_rows(src, dst, normalize=normalize)
        # fp32 -> fp16 may overflow: count the values that round to inf (one device -> host read)
        overflow = torch.zeros(1, dtype=torch.int32, device=self.device)
        engine.ingest_rows(src, dst, normalize=normalize, overflow=overflow)
        bad = int(overflow.item())
        if bad:
            raise ValueError(f"{bad} value(s) overflow fp16 (|x| >= 65520 after normalisation, or not finite); "
                             "nothing was added")
        return dst

    def _ingest_exact(self, src, dst32, dst, v_max=None):
        """Rows -> fp32 rows ``dst32`` (normalised in fp32 for cos) and their scan copy ``dst``: the rounding
        of the stored fp32 rows, so the two copies agree by construction."""
        src = src.to(self.device, non_blocking=True).float()
        if src.stride(1) != 1:
            src = src.contiguous()
        engine.ingest_rows_f32(src, dst32, normalize=self.normalize, v_max=v_max)
        self._scan_copy(dst32, dst)
        return dst32, dst

    def _scan_copy(self, rows32, dst):
        """The scan-format rounding of stored fp32 rows (no second normalisation; fp16 overflow refused)."""
        return self._ingest(rows32, dst, normalize=False)

    @classmethod
    def from_tensor(cls, emb, device="cuda", normalize=False, id_offset=0, chunk=1 << 18, dtype=torch.bfloat16,
                    exact=False):
        emb = torch.as_tensor(emb)
        t = cls(emb.shape[0], emb.shape[1], device=device, normalize=normalize, id_offset=id_offset, dtype=dtype,
                exact=exact)
        for s in range(0, emb.shape[0], chunk):
            t.append(emb[s : s + chunk])
        return t

    def encode_queries(self, q):
        """Query/user embeddings -> [B, ld] of the table's dtype under its similarity convention (exact
        tables: the fp32 rows; ``search`` derives their scan copy)."""
        q = torch.as_tensor(q)
        if q.dim() == 1:
            q = q.unsqueeze(0)
        if self.exact:
            out = torch.empty((q.shape[0], self.ld), dtype=torch.float32, device=self.device)
            return engine.ingest_rows_f32(q.to(self.device).float().contiguous(), out, normalize=self.normalize)
        out = torch.empty((q.shape[0], self.ld), dtype=self.dtype, device=self.device)
        return self._ingest(q, out)

    def search(self, queries, k, mask=None, algo=0, allow_short=False, want_f64=False, encoded=False,
               want_keys=False):
        """Top-k of queries against the resident rows.  Returns (scores, global ids[, scores64 | keys])."""
        if self.exact:
            return self._search_exact(queries, k, mask, algo, allow_short, want_f64, encoded, want_keys)[:-1]
        q = queries if encoded else self.encode_queries(queries)
        return engine.score_topk(q, self.data, k, mask=mask, id_offset=self.id_offset, algo=algo,
                                 allow_short=allow_short, want_f64=want_f64, n_items=self.n, D=self.ld,
                                 want_keys=want_keys)

    def _search_exact(self, queries, k, mask=None, algo=0, allow_short=False, want_f64=False, encoded=False,
                      want_keys=False):
        """``search`` of an exact table, plus the number of rows that went through the fallback."""
        if want_keys:
            raise ValueError("exact tables rank by float64 values: packed keys are not available")
        q = queries if encoded else self.encode_queries(queries)
        if q.dtype != torch.float32:
            raise TypeError("an exact table's encoded queries are its fp32 rows (encode_queries)")
        q_scan = torch.empty(q.shape, dtype=self.dtype, device=self.device)
        self._scan_copy(q, q_scan)
        s, i, d, n_fb = engine.score_topk_exact(q, q_scan, self.data32, self.data, k, self.v_max, mask=mask,
                                                id_offset=self.id_offset, algo=algo, allow_short=allow_short,
                                                n_items=self.n, D=self.ld)
        return ((s, i, d) if want_f64 else (s, i)) + (n_fb,)

    def dense_scores(self, queries, encoded=False):
        if self.exact:
            raise NotImplementedError("exact tables rank exactly but have no exact dense scores; use an "
                                      "EmbeddingTable without exact=True for dense score matrices")
        q = queries if encoded else self.encode_queries(queries)
        return engine.score_dense(q, self.data, n_items=self.n, D=self.ld)

    # ---- persistence: the `name=` analogue of generate_embeddings (ms_marco_eval.py:150-151) ----
    def save(self, path):
        blob = {"rows": self.rows.cpu(), "dim": self.dim, "normalize": self.normalize,
                "id_offset": self.id_offset, "dtype": _DTYPE_NAMES[self.dtype]}
        if self.exact:
            blob.update(exact=True, rows32=self.data32[: self.n].cpu(), v_max=float(self.v_max.item()))
        torch.save(blob, path)

    @classmethod
    def load(cls, path, device="cuda"):
        blob = torch.load(path)
        dtype = getattr(torch, blob.get("dtype", "bfloat16"))  # files written before fp16 tables: bf16
        exact = bool(blob.get("exact", False))  # files written before exact tables: not exact
        t = cls(blob["rows"].shape[0], blob["dim"], device=device, normalize=blob["normalize"],
                id_offset=blob["id_offset"], dtype=dtype, exact=exact)
        t.data[: blob["rows"].shape[0]].copy_(blob["rows"])
        if exact:
            t.data32[: blob["rows"].shape[0]].copy_(blob["rows32"])
            t.v_max.fill_(blob["v_max"])
        t.n = blob["rows"].shape[0]
        return t
