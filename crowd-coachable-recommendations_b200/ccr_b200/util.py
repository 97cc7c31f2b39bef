"""Top-k assignment over (lazy) score matrices: drop-in for the reference's
``rime_lite.util._assign_topk`` (src/rime_lite/util/__init__.py:117-155).

Same signature and return value -- a ``scipy.sparse.csr_matrix`` of ones, shape ``S.shape``,
exactly k entries per row with ``indices`` in top-k order -- but a score expression of the
hot-path shape ``LazyDense(U) @ LazyDense(V).T [+ prior_csr]`` is executed by the fused CUDA
kernel on a device-resident bf16 copy of V (uploaded once, not once per row batch as
score_array.py:226-227 does) and the [batch, N] float64 block is never materialised.

Deviations, documented in DESIGN.md: ``device`` and ``batch_size`` are accepted and ignored
(the work always runs on the table's GPU); the reference's unseeded ``rand * tie_breaker``
jitter (:139-140) is replaced by a deterministic lowest-column-first tie break.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sps
import torch

from . import _lib, engine
from .score_array import LazyScoreBase, auto_cast_lazy_score, dense_plan, fused_plan
from .table import EmbeddingTable

ROW_CHUNK = 8192


def _device_table_for(right, exact=False):
    """bf16 device table for the right factor ([D, N] LazyDenseMatrix), cached on the leaf so the
    row-batch slices of one expression (which share ``right``) upload it once.  ``exact``: an exact
    table (fp32 rows + scan copy, DESIGN.md section 6b), cached apart from the bf16 one.  Its scan copy is
    fp16, which needs far fewer candidates than bf16 for the same certified share, unless the factor
    holds values that fp16 cannot represent; the ranking is exact either way."""
    attr = "_ccr_table_exact" if exact else "_ccr_table"
    t = getattr(right, attr, None)
    if t is None:
        rows = torch.as_tensor(np.ascontiguousarray(right.c.T))
        if exact:
            big = rows.numel() and not bool(torch.isfinite(rows).all() and rows.abs().max() < EXACT_F16_LIMIT)
            t = EmbeddingTable.from_tensor(rows, dtype=torch.bfloat16 if big else torch.float16, exact=True)
        else:
            t = EmbeddingTable.from_tensor(rows)
        setattr(right, attr, t)
    return t


EXACT_F16_LIMIT = 32768.0  # factor values at or above this take a bf16 scan copy (fp16 overflows at 65520)


DENSE_CHUNK_ELEMS = 1 << 27  # dense score elements ranked per device pass (1 GB of float64)


def _topk_materialised(plan, k, want_scores):
    """Top-k of an already materialised dense score matrix (+ sparse prior) with the reference's
    ``as_tensor`` semantics -- the dense leaf keeps its dtype, adding the float64 CSR promotes to
    float64 (src/rime_lite/util/score_array.py:173-174,291-293).  float32 (and narrower) leaves,
    i.e. everything the reference's ``transform`` produces, run through the C ABI
    (``ccr_topk_dense_f32``: streaming exact top-k, priors merged as float64 overrides).  A float64
    leaf would need 64-bit score keys; that corner (never produced by the reference's own callers)
    is ranked by a stable device sort instead.  Ties -> lowest column either way."""
    if not torch.cuda.is_available():
        raise RuntimeError("ccr_b200 needs a CUDA device (no CPU path)")
    dev = torch.device("cuda")
    B, N = plan.shape
    if k > N:
        raise RuntimeError("selected index k out of range")
    ids = np.empty((B, k), dtype=np.int64)
    vals = np.empty((B, k), dtype=np.float64) if want_scores else None
    leaf = np.asarray(plan.dense.c)
    native = leaf.dtype in (np.float32, np.float16) and k <= _lib.MAX_K
    mask_all = None
    if native and plan.sparse is not None:
        mask_all = engine.SparseMask.from_scipy(plan.sparse, engine.MASK_ADD, dev)
        native = k + mask_all.max_row_nnz <= _lib.MAX_K
    rows_per = max(1, min(DENSE_CHUNK_ELEMS // max(1, N), 65535))
    for s in range(0, B, rows_per):
        e = min(B, s + rows_per)
        dense = torch.as_tensor(np.ascontiguousarray(leaf[s:e])).to(dev)
        if native:
            m = mask_all.rows(s, e) if mask_all is not None else None
            _, order, top = engine.topk_dense(dense.float(), k, mask=m)
            ids[s:e] = order.cpu().numpy()
            if want_scores:
                vals[s:e] = top.cpu().numpy()
            continue
        if plan.sparse is not None:
            coo = plan.sparse[s:e].tocoo()
            dense = dense.double()
            dense.index_put_((torch.as_tensor(coo.row, dtype=torch.int64, device=dev),
                              torch.as_tensor(coo.col, dtype=torch.int64, device=dev)),
                             torch.as_tensor(coo.data, dtype=torch.float64, device=dev), accumulate=True)
        top, order = torch.sort(dense, dim=1, descending=True, stable=True)
        ids[s:e] = order[:, :k].cpu().numpy()
        if want_scores:
            vals[s:e] = top[:, :k].double().cpu().numpy()
    return (ids, vals) if want_scores else ids


def topk_lazy(S, k, want_scores=False, algo=0, exact=False):
    """(ids [B,k] int64 numpy[, scores64 [B,k]]) for a fused-plan expression (factor pair: the
    fused kernel) or a materialised dense matrix (+ priors); None if S is neither.  ``exact``: a factor
    pair is ranked by its exact fp32 scores (DESIGN.md section 6b); a materialised matrix is already
    ranked exactly by its given values, so there it changes nothing."""
    plan = fused_plan(S)
    if plan is None:
        dplan = dense_plan(S)
        return _topk_materialised(dplan, k, want_scores) if dplan is not None else None
    B, N = plan.shape
    if k > N:
        raise RuntimeError("selected index k out of range")
    table = _device_table_for(plan.right, exact=exact)
    U = torch.as_tensor(np.ascontiguousarray(plan.left.c))
    ids = np.empty((B, k), dtype=np.int64)
    vals = np.empty((B, k), dtype=np.float64) if want_scores else None
    mask_all = None
    if plan.sparse is not None:
        mask_all = engine.SparseMask.from_scipy(plan.sparse, engine.MASK_ADD, table.device)
    for s in range(0, B, ROW_CHUNK):
        e = min(B, s + ROW_CHUNK)
        m = mask_all.rows(s, e) if mask_all is not None else None
        out = table.search(U[s:e], k, mask=m, algo=algo, want_f64=want_scores)
        ids[s:e] = out[1].cpu().numpy()
        if want_scores:
            vals[s:e] = out[2].cpu().numpy()
    return (ids, vals) if want_scores else ids


def _assign_topk(S, k, tie_breaker=1e-10, device="cpu", batch_size=None, exact=False):
    """Return a sparse matrix where each row contains k non-zero values (see module docstring);
    ``exact`` ranks a factor pair by its exact fp32 scores (``topk_lazy``)."""
    if not isinstance(S, LazyScoreBase):
        S = auto_cast_lazy_score(S)
    indices = topk_lazy(S, k, exact=exact)
    if indices is None:
        raise NotImplementedError(
            f"_assign_topk: expression {S!r} is outside the accelerated score-and-rank path "
            "(supported: LazyDense @ LazyDense.T [+/- sparse priors], LazyDense [+/- sparse priors]); "
            "see DESIGN.md 'out of scope'")
    return sps.csr_matrix(
        (np.ones(indices.size), np.ravel(indices), np.arange(0, indices.size + 1, indices.shape[1])),
        shape=S.shape,
    )


assign_topk = _assign_topk


def _argsort(S, tie_breaker=1e-10, device="cpu", exact=False):
    """Drop-in for ``rime_lite.util._argsort`` (src/rime_lite/util/__init__.py:158-184): global flat
    argsort of the whole score matrix, best score first, returned as ``(row_idx, col_idx)``.

    The fp32 score matrix is produced on the device (``ccr_score_dense_f32``: the TMA + tcgen05 pipeline
    with a store epilogue for tiles of >= 2^20 scores) -- or uploaded, when the expression is an already
    materialised dense matrix -- and ordered by ``ccr_argsort_scores_f32``, an LSD radix sort over
    float64-ordered keys with the sparse priors merged in float64 like the reference's promotion.
    Ties are ordered by flat position (the reference adds unseeded jitter).  ``exact``: a factor pair is
    scored by its exact fp32 scores (``ccr_score_dense_exact`` on the exact table ``_assign_topk(exact=True)``
    uses, DESIGN.md section 6b); a materialised matrix is ordered by its given values either way."""
    if not isinstance(S, LazyScoreBase):
        S = auto_cast_lazy_score(S)
    plan = fused_plan(S)
    if plan is not None:
        table = _device_table_for(plan.right, exact=exact)
        dense = table.dense_scores(torch.as_tensor(np.ascontiguousarray(plan.left.c)), exact=exact)
        sparse = plan.sparse
    else:
        dplan = dense_plan(S)
        if dplan is None or np.asarray(dplan.dense.c).dtype not in (np.float32, np.float16):
            raise NotImplementedError(f"_argsort: expression {S!r} is outside the accelerated score-and-rank path")
        if not torch.cuda.is_available():
            raise RuntimeError("ccr_b200 needs a CUDA device (no CPU path)")
        dense = torch.as_tensor(np.ascontiguousarray(dplan.dense.c)).to("cuda").float()
        sparse = dplan.sparse
    mask = engine.SparseMask.from_scipy(sparse, engine.MASK_ADD, dense.device) if sparse is not None else None
    rows, cols = engine.argsort_scores(dense, mask)
    return rows.cpu().numpy(), cols.cpu().numpy()


argsort = _argsort


def transform_scores(all_emb, i_to_ptr, j_to_ptr, sim_type=None):
    """The users x items score matrix of ``BertBPR.transform`` (src/ccrec/models/bbpr.py:528-550) as a
    lazy factor pair instead of a dense host matrix: ``all_emb[i_to_ptr] @ all_emb[j_to_ptr].T``, with
    both sides L2-normalised first (``F.normalize``, eps 1e-12) when CCREC_SIM_TYPE is ``cos``.
    ``+ D.prior_score``, ``_assign_topk`` and ``evaluate_item_rec`` then run through the fused kernel;
    nothing of size users x items is ever materialised."""
    import os

    from .score_array import LazyDenseMatrix

    if sim_type is None:
        sim_type = os.environ["CCREC_SIM_TYPE"]  # KeyError when unset, like bbpr.py:538
    emb = torch.as_tensor(all_emb).detach().float().cpu()
    users, items = emb[torch.as_tensor(np.asarray(i_to_ptr))], emb[torch.as_tensor(np.asarray(j_to_ptr))]
    if sim_type == "cos":
        users = torch.nn.functional.normalize(users, p=2, dim=1)
        items = torch.nn.functional.normalize(items, p=2, dim=1)
    return LazyDenseMatrix(users.numpy()) @ LazyDenseMatrix(items.numpy()).T
