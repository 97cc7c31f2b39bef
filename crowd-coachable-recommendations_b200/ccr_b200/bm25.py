"""Drop-ins for the reference's lexical baseline: ``BM25`` (scripts/bm_25.py:9-45) and
``ranking_bm25`` (scripts/ms_marco_eval.py:165-186).

Tokenisation, vocabulary and idf stay sklearn's ``TfidfVectorizer(norm=None, smooth_idf=False)``
on the host, exactly as in the reference (text processing is not the hot path).  What moves to
the device is everything per query: the reference slices the CSC count matrix, builds dense
[N, T] numerators/denominators with scipy, sums them, then ``ranking_bm25`` full-sorts the N
scores for 1001 outputs -- 21 min for 3,452 NQ queries (SURVEY.md §6).  Here the postings live
on the device with their query-independent BM25 values precomputed at ``fit``/``cache`` time
(``ccr_bm25_build_impacts``), and one fused kernel per query batch accumulates the scores in
shared memory and keeps the top-k (``ccr_bm25_topk``).  There is no CPU scoring path.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .engine import _require_cuda, _stream_ptr, workspace  # noqa: F401

RANKING_TOPN = 1001  # scripts/ms_marco_eval.py:182
QUERY_CHUNK = 4096   # queries per fused call
WARP_KERNEL_MAX_TERMS = 32  # libccr_b200: kBmwMaxTerms
MAX_QUERY_TERMS = 512
HEAD_DF_FRACTION = 0.25     # terms present in at least this share of the docs also get a dense float64 row
HEAD_MAX_TERMS = 64
HEAD_MAX_BYTES = 4 << 30


class BM25(object):
    """Same constructor, ``fit``, ``cache`` and ``transform`` as scripts/bm_25.py:9-45."""

    def __init__(self, b=0.75, k1=1.6, device="cuda", head_df_fraction=HEAD_DF_FRACTION):
        """``head_df_fraction``: vocabulary terms that occur in at least this share of the cached
        documents (stop words) additionally get a dense float64 row on the device, which the kernels
        add with coalesced loads instead of walking the posting list (``None`` / 0: postings only).
        The scores are bit-identical either way."""
        from sklearn.feature_extraction.text import TfidfVectorizer

        self.vectorizer = TfidfVectorizer(norm=None, smooth_idf=False)
        self.b = b
        self.k1 = k1
        self.device = torch.device(device)
        self.head_df_fraction = head_df_fraction
        self._impacts_stale = True
        self._head_slot = self._head_rows = None

    # ---- reference API -------------------------------------------------------------------
    def fit(self, X):
        """Fit IDF to documents X (bm_25.py:15-20)."""
        self.vectorizer.fit(X)
        self.cache(X)
        self.avdl = self.last_len_X.mean()
        self._impacts_stale = True
        return self

    def cache(self, X):
        """Count matrix of X as device-resident postings (bm_25.py:22-25)."""
        csc = self._counts(X).tocsc()
        csc.sort_indices()
        self.last_csc_X = csc
        self.last_len_X = np.asarray(csc.sum(1)).ravel()
        if csc.shape[0] >= (1 << 31) - 512:
            raise ValueError("BM25: more than 2^31 documents")
        if csc.nnz and csc.data.max() >= (1 << 24):
            raise ValueError("BM25: a term count >= 2^24 is not exactly representable as float32")
        if self.device.type != "cuda":
            raise RuntimeError("ccr_b200.BM25 needs a CUDA device (no CPU path)")
        dev = self.device
        self._indptr = torch.as_tensor(csc.indptr.astype(np.int64)).to(dev)
        self._docs = torch.as_tensor(csc.indices.astype(np.int32)).to(dev)
        self._tf = torch.as_tensor(csc.data.astype(np.float32)).to(dev)
        self._val = torch.empty(csc.nnz, dtype=torch.float64, device=dev)
        self._impacts_stale = True
        return self

    def transform(self, q, X=None):
        """BM25 between query q and the cached documents -> float64 ndarray [N] (bm_25.py:27-45)."""
        if X is not None:
            self.cache(X)
        return self.scores([q])[0].cpu().numpy()

    # ---- batched device API ----------------------------------------------------------------
    def _counts(self, texts):
        from sklearn.feature_extraction.text import CountVectorizer

        return CountVectorizer.transform(self.vectorizer, texts)  # = super(TfidfVectorizer, v).transform

    @property
    def n_docs(self):
        return self.last_csc_X.shape[0]

    def _ensure_impacts(self):
        if not self._impacts_stale:
            return
        b, k1, avdl = self.b, self.k1, self.avdl
        doc_norm = k1 * (1 - b + b * self.last_len_X / avdl)          # bm_25.py:41
        idf = self.vectorizer._tfidf.idf_ - 1.0                       # bm_25.py:42-44
        dev = self.device
        d_norm = torch.as_tensor(np.ascontiguousarray(doc_norm, dtype=np.float64)).to(dev)
        d_idf = torch.as_tensor(np.ascontiguousarray(idf, dtype=np.float64)).to(dev)
        n_terms, nnz = self._indptr.numel() - 1, self._docs.numel()
        with torch.cuda.device(dev):
            rc = _lib.lib().ccr_bm25_build_impacts(self._indptr.data_ptr(), self._docs.data_ptr(), self._tf.data_ptr(),
                                                   d_idf.data_ptr(), d_norm.data_ptr(), float(k1), n_terms, nnz,
                                                   self._val.data_ptr(), _stream_ptr(dev))
        _lib.check(rc)
        self._build_head_rows()
        torch.cuda.current_stream(dev).synchronize()  # d_norm / d_idf are released on return
        self._impacts_stale = False

    def head_terms(self):
        """Vocabulary ids of the terms that get a dense row: df >= head_df_fraction * N, the most frequent
        first, at most HEAD_MAX_TERMS of them and HEAD_MAX_BYTES of rows."""
        N = self.n_docs
        if not self.head_df_fraction or N == 0:
            return np.zeros(0, np.int32)
        df = np.diff(self.last_csc_X.indptr)
        cand = np.nonzero(df >= max(1.0, self.head_df_fraction * N))[0]
        cand = cand[np.argsort(-df[cand], kind="stable")]
        pitch = int(_lib.lib().ccr_bm25_head_row_pitch(N))
        limit = min(HEAD_MAX_TERMS, HEAD_MAX_BYTES // max(1, pitch * 8))
        return np.ascontiguousarray(cand[:limit], dtype=np.int32)

    def _build_head_rows(self):
        self._head_slot = self._head_rows = None
        terms = self.head_terms()
        if terms.size == 0:
            return
        dev, N = self.device, self.n_docs
        L = _lib.lib()
        n_terms = self._indptr.numel() - 1
        d_terms = torch.as_tensor(terms).to(dev)
        slot = torch.empty(n_terms, dtype=torch.int32, device=dev)
        rows = torch.empty((terms.size, int(L.ccr_bm25_head_row_pitch(N))), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = L.ccr_bm25_build_head_rows(self._indptr.data_ptr(), self._docs.data_ptr(), self._val.data_ptr(),
                                            d_terms.data_ptr(), int(terms.size), n_terms, N, slot.data_ptr(),
                                            rows.data_ptr(), _stream_ptr(dev))
        _lib.check(rc)
        torch.cuda.current_stream(dev).synchronize()  # d_terms is released on return
        self._head_slot, self._head_rows = slot, rows

    def _head_ptrs(self):
        if self._head_rows is None:
            return None, None
        return self._head_slot.data_ptr(), self._head_rows.data_ptr()

    def encode_queries(self, texts):
        """texts -> (q_indptr int64 [B+1], q_terms int32, longest row): the DISTINCT vocabulary terms
        of every query in ascending id order (the reference only uses ``q.indices``, bm_25.py:38)."""
        m = self._counts(list(texts)).tocsr()
        m.sort_indices()
        longest = int(np.diff(m.indptr).max()) if m.shape[0] else 0
        if longest > MAX_QUERY_TERMS:
            raise ValueError(f"BM25: a query has {longest} distinct terms (limit {MAX_QUERY_TERMS})")
        return m.indptr.astype(np.int64), m.indices.astype(np.int32), longest

    def _device_queries(self, texts):
        indptr, terms, longest = self.encode_queries(texts)
        dev = self.device
        d_indptr = torch.as_tensor(indptr).to(dev)
        d_terms = torch.as_tensor(terms if terms.size else np.zeros(1, np.int32)).to(dev)
        return d_indptr, d_terms, longest

    def scores(self, texts):
        """Dense float64 [B, N] BM25 scores on the device (``transform`` for a batch)."""
        self._ensure_impacts()
        B, N, dev = len(texts), self.n_docs, self.device
        out = torch.empty((B, N), dtype=torch.float64, device=dev)
        if B == 0 or N == 0:
            return out
        d_indptr, d_terms, longest = self._device_queries(texts)
        with torch.cuda.device(dev):
            rc = _lib.lib().ccr_bm25_scores_f64(self._indptr.data_ptr(), self._docs.data_ptr(), self._val.data_ptr(),
                                                *self._head_ptrs(), d_indptr.data_ptr(), d_terms.data_ptr(), longest, B, N,
                                                out.data_ptr(), N, _stream_ptr(dev))
        _lib.check(rc)
        return out

    def topk(self, texts, k):
        """Per query the k best documents ranked as float32 like ``ranking_bm25``
        (ms_marco_eval.py:179-181): (scores float32 [B,k] descending, positions int64 [B,k]),
        ties -> lowest position."""
        self._ensure_impacts()
        B, N, dev = len(texts), self.n_docs, self.device
        k = int(k)
        out_s = torch.empty((B, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
        L = _lib.lib()
        if k > N:  # same error as Tensor.topk; also raised by the C ABI for B > 0
            raise RuntimeError(f"selected index k out of range (k={k} > n={N})")
        for s in range(0, B, QUERY_CHUNK):
            e = min(B, s + QUERY_CHUNK)
            indptr, terms, _ = self.encode_queries(texts[s:e])
            lengths = np.diff(indptr)
            # the library picks its kernel per call from the longest query: the barrier-free warp-private
            # kernel up to WARP_KERNEL_MAX_TERMS distinct terms, the block-wide one beyond -- so the rare
            # long queries (whole passages) go in a call of their own and do not slow the short ones down
            short = np.nonzero(lengths <= WARP_KERNEL_MAX_TERMS)[0]
            long_ = np.nonzero(lengths > WARP_KERNEL_MAX_TERMS)[0]
            for rows in (short, long_):
                if rows.size == 0:
                    continue
                whole = rows.size == e - s
                sub_ptr = indptr if whole else np.concatenate([[0], np.cumsum(lengths[rows])]).astype(np.int64)
                sub_terms = terms if whole else (np.concatenate([terms[indptr[r]:indptr[r + 1]] for r in rows])
                                                 if lengths[rows].sum() else np.zeros(0, np.int32))
                d_indptr = torch.as_tensor(sub_ptr).to(dev)
                d_terms = torch.as_tensor(sub_terms if sub_terms.size else np.zeros(1, np.int32)).to(dev)
                n_q = int(rows.size)
                res_s = out_s[s:e] if whole else torch.empty((n_q, k), dtype=torch.float32, device=dev)
                res_i = out_i[s:e] if whole else torch.empty((n_q, k), dtype=torch.int64, device=dev)
                with torch.cuda.device(dev):
                    ws = workspace.get(dev, L.ccr_bm25_topk_workspace_bytes(n_q, N, k))
                    rc = L.ccr_bm25_topk(self._indptr.data_ptr(), self._docs.data_ptr(), self._val.data_ptr(),
                                         *self._head_ptrs(), d_indptr.data_ptr(), d_terms.data_ptr(),
                                         int(lengths[rows].max()), n_q, N, k,
                                         res_s.data_ptr(), res_i.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(dev))
                _lib.check(rc)
                if not whole:
                    at = torch.as_tensor(rows + s, device=dev)
                    out_s.index_copy_(0, at, res_s)
                    out_i.index_copy_(0, at, res_i)
        return out_s, out_i


def ranking_bm25(corpus, queries, device="cuda"):
    """scripts/ms_marco_eval.py:165-186: ``{qid: {pid: score}}`` with the best 1001 (or N)
    passages per query in descending float32 BM25 order."""
    ranking_profile = {}
    model = BM25(b=0.75, k1=1.2, device=device)
    print("Fitting BM-25 model")
    model.fit(list(corpus.values()))
    print("Retrieval with BM-25 model")
    queries_ids = list(queries.keys())
    corpus_ids = list(corpus.keys())
    if not queries_ids:
        return ranking_profile
    k = min(RANKING_TOPN, len(corpus_ids))
    scores, order = model.topk([queries[q] for q in queries_ids], k)
    scores, order = scores.cpu().numpy(), order.cpu().numpy()
    corpus_arr = np.asarray(corpus_ids, dtype=object)
    for step, qid in enumerate(queries_ids):
        ranking_profile[qid] = dict(zip(corpus_arr[order[step]].tolist(), scores[step].tolist()))
    return ranking_profile
