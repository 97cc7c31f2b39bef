"""Drop-in for the reference's dense retrieval entry point.

``ranking(corpus, queries, embedding_func, batch_size, block_dict=None)`` keeps the signature,
inputs and return value of scripts/ms_marco_eval.py:189-235 -- ``{qid: {pid: score}}`` holding
the best 1001 (or N) passages per query in descending score order, block-listed passages
carrying -1e6 -- but never builds the Q x N host matrix nor sorts full rows: embeddings go
straight into a device-resident bf16 table and one fused kernel does score + mask + top-k.

Deliberate deviations (documented in DESIGN.md): scores come from bf16-rounded embeddings with
fp32 accumulation (the reference's GPU path under autocast is fp16-in/fp16-out,
scripts/al_0_rank.py:125); exact ties are ordered by corpus position (reference: unspecified).
``table_dtype=torch.float16`` rounds the embeddings to fp16 instead, the reference's own operand
format, so the ranking matches its autocast run up to accumulation order; the scores stay fp32.
"""
from __future__ import annotations

import math
import os
from collections.abc import Mapping

import numpy as np
import torch

from . import engine
from .table import EmbeddingTable, check_table_dtype

RANKING_TOPN = 1001  # scripts/ms_marco_eval.py:230
BLOCK_VALUE = -1e6   # scripts/ms_marco_eval.py:227
QUERY_CHUNK = 8192   # query rows per fused call (bounds workspace and the [B,k] result)


def cos_sim(a: torch.Tensor, b: torch.Tensor):
    """scripts/ms_marco_eval.py:155-162 on the device path: fp32 normalise -> bf16 -> dense scores."""
    a = torch.as_tensor(a)
    b = torch.as_tensor(b)
    if a.dim() == 1:
        a = a.unsqueeze(0)
    if b.dim() == 1:
        b = b.unsqueeze(0)
    t = EmbeddingTable.from_tensor(b, normalize=True)
    return t.dense_scores(a)


def generate_embeddings(data_indices, data_dic, embedding_func, batch_size, embedding_size=768, name=None):
    """Reference-compatible signature (scripts/ms_marco_eval.py:123-152): returns a CPU fp32
    tensor.  Kept for callers that want the host copy; ``ranking`` uses
    ``generate_embeddings_device`` instead."""
    out = []
    with torch.no_grad():
        for step in range(math.ceil(len(data_indices) / batch_size)):
            idx = data_indices[step * batch_size : (step + 1) * batch_size]
            out.append(torch.as_tensor(embedding_func([data_dic[i] for i in idx])).to("cpu"))
    emb = torch.vstack(out) if out else torch.zeros(0, embedding_size)
    if name is not None:
        torch.save(emb, name)
    return emb


def generate_embeddings_device(data_indices, data_dic, embedding_func, batch_size, normalize=False,
                               device="cuda", id_offset=0, name=None, dtype=torch.bfloat16, exact=False):
    """Encoder batches -> device bf16 (or ``dtype``) table without the host round trip (SURVEY.md §8f-1);
    ``exact``: the table also keeps the fp32 rows and searches rank exactly (DESIGN.md section 6b)."""
    check_table_dtype(dtype)
    table = None
    with torch.no_grad():
        for step in range(math.ceil(len(data_indices) / batch_size)):
            idx = data_indices[step * batch_size : (step + 1) * batch_size]
            emb = torch.as_tensor(embedding_func([data_dic[i] for i in idx]))
            if table is None:
                table = EmbeddingTable(len(data_indices), emb.shape[1], device=device, normalize=normalize,
                                       id_offset=id_offset, dtype=dtype, exact=exact)
            table.append(emb)
    if table is None:
        table = EmbeddingTable(0, 768, device=device, normalize=normalize, id_offset=id_offset, dtype=dtype,
                               exact=exact)
    if name is not None:
        table.save(name)
    return table


def build_block_mask(queries_ids, corpus_ids, block_dict, device):
    """block_dict {qid: [pid, ...]} -> SparseMask(set -1e6).  Mirrors ms_marco_eval.py:225-227
    including the "block id not found" assertion, with the pid->position index built once and ONE
    lookup over all block lists instead of one index build + lookup per query."""
    import pandas as pd

    from itertools import chain

    index = pd.Index(corpus_ids)
    blocks = [block_dict[qid] for qid in queries_ids]  # KeyError for a query without an entry, like :225
    lengths = [len(b) for b in blocks]
    ind = index.get_indexer(list(chain.from_iterable(blocks))) if sum(lengths) else np.zeros(0, dtype=np.int64)
    assert -1 not in ind, "block id not found"
    return engine.SparseMask.from_flat(lengths, ind, len(corpus_ids), BLOCK_VALUE, engine.MASK_SET, device)


class RankingProfile(Mapping):
    """The ``{qid: {pid: score}}`` result of ``ranking`` held as the two [Q, k] arrays the kernels
    produce (scores float32, corpus positions int64).  It behaves like the reference's dict -- keys in
    query order, ``profile[qid]`` is a dict in descending score order, ``==`` against a dict, pickling
    yields a plain dict (``rank_step`` saves ``to_dict()`` so ``ranking_profile.pt`` keeps the reference's
    format and loads under torch.load's weights-only default) --
    but a row's dict is only built when somebody asks for it (9,862 x 1,001 entries cost 1.2 s up
    front, SURVEY.md section 8f-2); MRR and candidate selection read the arrays directly."""

    def __init__(self, queries_ids, corpus_ids, scores, order):
        self.queries_ids = list(queries_ids)
        self.corpus_ids = corpus_ids if isinstance(corpus_ids, np.ndarray) else np.asarray(list(corpus_ids), dtype=object)
        self.scores = np.asarray(scores)
        self.order = np.asarray(order)
        self._row_of = {qid: i for i, qid in enumerate(self.queries_ids)}
        self._cache = {}

    def __getitem__(self, qid):
        row = self._cache.get(qid)
        if row is None:
            i = self._row_of[qid]  # KeyError like a dict
            row = dict(zip(self.corpus_ids[self.order[i]].tolist(), self.scores[i].tolist()))
            self._cache[qid] = row
        return row

    def __iter__(self):
        return iter(self.queries_ids)

    def __len__(self):
        return len(self.queries_ids)

    def __contains__(self, qid):
        return qid in self._row_of

    def top_ids(self, qid, n):
        """The first ``n`` passage ids of a query without building its dict."""
        return self.corpus_ids[self.order[self._row_of[qid], :n]].tolist()

    def to_dict(self):
        return {qid: self[qid] for qid in self.queries_ids}

    def __reduce__(self):
        return (dict, (self.to_dict(),))

    def __repr__(self):
        return f"RankingProfile({len(self)} queries x {self.order.shape[1] if self.order.ndim == 2 else 0} passages)"


def ranking_tensors(query_table, passage_table, k, mask=None, algo=0):
    """Core of ``ranking``: resident tables -> (scores [Q,k] f32, positions [Q,k] i64) on the host."""
    Q = len(query_table)
    scores = np.empty((Q, k), dtype=np.float32)
    order = np.empty((Q, k), dtype=np.int64)
    for s in range(0, Q, QUERY_CHUNK):
        e = min(Q, s + QUERY_CHUNK)
        m = mask.rows(s, e) if mask is not None else None
        q = query_table.data32 if query_table.exact else query_table.data
        sc, ids = passage_table.search(q[s:e], k, mask=m, algo=algo, encoded=True)
        scores[s:e] = sc.cpu().numpy()
        order[s:e] = ids.cpu().numpy()
    return scores, order


def ranking(corpus, queries, embedding_func, batch_size, block_dict=None, device="cuda", algo=0,
            table_dtype=torch.bfloat16, exact=False):
    """``table_dtype``: element type of the device tables, bf16 (default) or fp16 (the reference's
    autocast operand format); scores are fp32 either way.  ``exact``: rank by the exact fp32 scores of the
    reference's CPU path (DESIGN.md section 6b); ``table_dtype`` is then the format of the scan copy."""
    check_table_dtype(table_dtype)
    sim = os.environ["CCREC_SIM_TYPE"]  # KeyError when unset, like ms_marco_eval.py:212
    normalize = sim == "cos"
    queries_ids, corpus_ids = list(queries.keys()), list(corpus.keys())
    q_table = generate_embeddings_device(queries_ids, queries, embedding_func, batch_size, normalize, device,
                                         dtype=table_dtype, exact=exact)
    p_table = generate_embeddings_device(corpus_ids, corpus, embedding_func, batch_size, normalize, device,
                                         dtype=table_dtype, exact=exact)
    if len(queries_ids) == 0:
        return {}
    mask = None
    if block_dict is not None:
        print("using block_dict")
        mask = build_block_mask(queries_ids, corpus_ids, block_dict, p_table.device)
    k = min(RANKING_TOPN, len(corpus_ids))
    scores, order = ranking_tensors(q_table, p_table, k, mask, algo=algo)
    return RankingProfile(queries_ids, corpus_ids, scores, order)


def qrels_csr(queries_ids, corpus_ids, qrels):
    """Relevant corpus positions (qrels score > 0) per query as CSR (indptr int64 [Q+1], sorted int64
    positions); passages outside the corpus are ignored like BEIR ignores unknown doc ids."""
    pos = corpus_ids if isinstance(corpus_ids, dict) else {pid: i for i, pid in enumerate(corpus_ids)}
    indptr, rel = [0], []
    for qid in queries_ids:
        hits = sorted(pos[p] for p, s in qrels.get(qid, {}).items() if s > 0 and p in pos)
        rel.extend(hits)
        indptr.append(len(rel))
    return np.asarray(indptr, dtype=np.int64), np.asarray(rel, dtype=np.int64)


def mrr_at_k(order, corpus_ids, queries_ids, qrels, k_values=(1, 5, 10, 100), device="cuda"):
    """MRR@k of a ranking given as positions [Q, k] (descending), the metric scripts/al_0_rank.py:130-133
    obtains from BEIR's ``EvaluateRetrieval.evaluate_custom(qrels, results, k_values, metric="mrr")``
    (third party, unvendored and unpinned by the reference; its published algorithm): per query the
    reciprocal rank of the first passage with qrels score > 0 inside the top k is summed, the sum is
    divided by ``len(qrels)`` and rounded to 5 digits.  The first-hit scan runs on the device
    (``ccr_first_hit_rank``), one warp per query (SURVEY.md section 8f-2)."""
    order_t = order if isinstance(order, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(order), dtype=torch.int64)
    if not order_t.is_cuda:
        order_t = order_t.to(device)
    indptr, rel = qrels_csr(queries_ids, corpus_ids, qrels)
    first = engine.first_hit_rank(order_t, indptr, rel).cpu().numpy().astype(np.float64)
    n = max(1, len(qrels))
    out = {}
    for k in k_values:
        hit = (first > 0) & (first <= k)
        out[f"MRR@{k}"] = round(float(np.sum(1.0 / first[hit])) / n, 5)
    return out


def ranking_sharded(corpus, queries, embedding_func, batch_size, block_dict=None, group=None, device=None,
                    index_cls=None, table_dtype=torch.bfloat16, exact=False):
    """``ranking`` with the passage table row-sharded over the ranks of a torch.distributed group
    (one process per GPU): every rank encodes the queries and ONLY its own contiguous slice of the
    corpus (``shard_bounds``) straight into its device shard -- the encoder pass, which dominates the
    reference's wall clock, is split G ways and no rank ever holds the whole table -- then the
    fused local top-k, one all-gather and the G-way merge produce the global result.  Every rank
    returns the same ``{qid: {pid: score}}`` as the single-table call (``table_dtype`` and ``exact`` as in
    ``ranking``)."""
    from .dist import ShardedIndex

    check_table_dtype(table_dtype)
    sim = os.environ["CCREC_SIM_TYPE"]  # KeyError when unset, like ms_marco_eval.py:212
    normalize = sim == "cos"
    queries_ids, corpus_ids = list(queries.keys()), list(corpus.keys())
    if len(queries_ids) == 0:
        return {}
    with torch.no_grad():
        q_emb = torch.cat([torch.as_tensor(embedding_func([queries[i] for i in queries_ids[s:s + batch_size]]))
                           for s in range(0, len(queries_ids), batch_size)])
        index = (index_cls or ShardedIndex)(len(corpus_ids), q_emb.shape[1], normalize=normalize, device=device,
                                            group=group, dtype=table_dtype, exact=exact)
        for s in range(index.lo, index.hi, batch_size):
            e = min(index.hi, s + batch_size)
            index.add_local(torch.as_tensor(embedding_func([corpus[i] for i in corpus_ids[s:e]])))
    mask = None
    if block_dict is not None:
        print("using block_dict")
        mask = build_block_mask(queries_ids, corpus_ids, block_dict, index.device)
    k = min(RANKING_TOPN, len(corpus_ids))
    scores = np.empty((len(queries_ids), k), dtype=np.float32)
    order = np.empty((len(queries_ids), k), dtype=np.int64)
    for s in range(0, len(queries_ids), QUERY_CHUNK):
        e = min(len(queries_ids), s + QUERY_CHUNK)
        sc, ids, _ = index.search(q_emb[s:e], k, mask=mask.rows(s, e) if mask is not None else None)
        scores[s:e] = sc.cpu().numpy()
        order[s:e] = ids.cpu().numpy()
    return RankingProfile(queries_ids, corpus_ids, scores, order)
