"""``evaluate_item_rec`` / ``evaluate_assigned`` with the reference's outputs
(src/rime_lite/metrics/__init__.py:51-89).  The reference re-evaluates the whole score matrix
in row batches to compute ``obj_mean`` (:77, ``_sum`` :26-29); here the fused kernel already
returns the float64 value of every assigned entry, so ``obj_mean`` is O(B*k)."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sps

from .util import topk_lazy, _assign_topk
from .score_array import LazyScoreBase, auto_cast_lazy_score


def perplexity(x):
    x = np.ravel(x) / x.sum()
    return float(np.exp(-x @ np.log(np.where(x > 0, x, 1e-10))))


def evaluate_assigned(target_csr, assigned_csr, score_mat=None, axis=None, min_total_recs=0, device="cpu",
                      _assigned_score_sum=None):
    target_csr = sps.csr_matrix(target_csr)
    assigned_csr = sps.csr_matrix(assigned_csr)
    hits = target_csr.multiply(assigned_csr)
    hit_axis = np.asarray(hits.sum(axis=axis)) if axis is not None else hits.sum()
    assigned_sum_0 = np.asarray(assigned_csr.sum(axis=0))
    assigned_sum_1 = np.asarray(assigned_csr.sum(axis=1))
    min_total_recs = max(min_total_recs, assigned_sum_0.sum())
    out = {
        "prec": np.sum(hit_axis) / min_total_recs,
        "recs/user": assigned_sum_1.mean(),
        "item_cov": (assigned_sum_0 > 0).mean(),
        "item_ppl": perplexity(assigned_sum_0),
        "user_cov": (assigned_sum_1 > 0).mean(),
        "user_ppl": perplexity(assigned_sum_1),
    }
    if _assigned_score_sum is not None:
        out["obj_mean"] = float(_assigned_score_sum / min_total_recs)
    elif score_mat is not None:
        raise NotImplementedError("obj_mean needs the assigned scores; call evaluate_item_rec")
    if axis is not None:
        ideal = np.ravel(target_csr.sum(axis=axis))
        out["recall"] = (np.ravel(hit_axis) / np.fmax(1, ideal)).mean()
    return out


def evaluate_item_rec(target_csr, score_mat, topk, device="cpu", exact=False, **kw):
    S = score_mat if isinstance(score_mat, LazyScoreBase) else auto_cast_lazy_score(score_mat)
    res = topk_lazy(S, topk, want_scores=True, exact=exact)
    if res is None:
        _assign_topk(S, topk)  # raises the descriptive NotImplementedError
    ids, vals = res
    assigned = sps.csr_matrix(
        (np.ones(ids.size), np.ravel(ids), np.arange(0, ids.size + 1, ids.shape[1])), shape=S.shape)
    return evaluate_assigned(target_csr, assigned, S, axis=1, device=device, _assigned_score_sum=vals.sum())
