"""fp16-operand references and agreement metrics for the fp16 table tests (test infrastructure).

The oracle's arbiters round their operands to bf16 (``round_bf16=True``).  An fp16 table rounds to
IEEE binary16 instead; the same arbiters give its reference when they are handed operands that are
already fp16-rounded -- after the fp32 L2 normalisation for ``sim == "cos"``, exactly where the oracle
rounds -- with their own rounding switched off.

The metrics compare a ranking with the reference's REAL GPU output (tests/golden/ranking_cuda_autocast_*:
unmodified ms_marco_eval.ranking under torch.cuda.amp.autocast(), fp16 scores):
* score equality: our score at a rank, rounded to fp16, equals the golden's score at that rank (blocked
  positions carry -1e6 on both sides);
* tie-aware positions: our id at a rank lies in the golden's group of ids that share that rank's fp16
  score -- the reference's sort is unstable inside such a group, so any member is its answer;
* ordered top-2: the first two ids, in order (the pair al_0_rank.py:172 sends to labellers).
"""
import numpy as np
import torch

from oracle import ccr_oracle as O


def fp16_operands(Q, P, sim="dot"):
    """What an fp16 table stores: fp32 (L2-normalised for cos) rows rounded to fp16, widened to fp32."""
    Q = torch.as_tensor(Q).float()
    P = torch.as_tensor(P).float()
    if sim == "cos":
        Q, P = O.normalize_rows_ref(Q), O.normalize_rows_ref(P)
    return Q.half().float(), P.half().float()


def score_topk_ref_f16(Q, P, k, mask=None, mode=O.MASK_NONE, sim="dot", **kw):
    """``O.score_topk_ref`` with fp16 instead of bf16 operand rounding."""
    Qh, Ph = fp16_operands(Q, P, sim)
    return O.score_topk_ref(Qh, Ph, k, mask=mask, mode=mode, sim="dot", round_bf16=False, **kw)


def full_scores_ref_f16(Q, P, mask=None, mode=O.MASK_NONE, sim="dot"):
    """``O.full_scores_ref`` with fp16 instead of bf16 operand rounding."""
    Qh, Ph = fp16_operands(Q, P, sim)
    return O.full_scores_ref(Qh, Ph, mask=mask, mode=mode, sim="dot", round_bf16=False)


def golden_agreement(scores, order, g_scores, g_order):
    """(score-equal share, tie-aware position share, share of rows with the same ordered top-2) of a
    ranking (scores [Q,k] float, corpus positions [Q,k]) against a reference-GPU golden."""
    scores = np.asarray(scores, dtype=np.float32)
    order = np.asarray(order)
    live = g_scores > -1e6
    ours16 = scores.astype(np.float16).astype(np.float32)
    score_eq = np.where(live, ours16 == g_scores, scores == g_scores).mean()
    agree = 0
    for b in range(order.shape[0]):
        groups = {}
        for s_, i_ in zip(g_scores[b], g_order[b]):
            groups.setdefault(float(s_), set()).add(int(i_))
        agree += sum(int(order[b, r]) in groups[float(g_scores[b, r])] for r in range(order.shape[1]))
    tie_aware = agree / order.size
    top2 = (order[:, :2] == g_order[:, :2]).all(1).mean()
    return float(score_eq), float(tie_aware), float(top2)


def emulate_ranking(case, rnd, k):
    """The ranking of a CUDA_RANKING_CASES case from operands rounded by ``rnd`` with the products summed
    in float64 (no accumulation-order effects), block-listed positions at -1e6, stable descending sort,
    first k.  Returns (scores float32 [Q,k], positions [Q,k])."""
    c = case
    pos = {p: i for i, p in enumerate(c["corpus"])}
    qpos = [int(v.split("#")[1]) for v in c["queries"].values()]
    T = torch.as_tensor(c["table"])
    n = len(c["corpus"])
    P, Q = T[:n].float(), T[qpos].float()
    if c["sim_type"] == "cos":
        P, Q = O.normalize_rows_ref(P), O.normalize_rows_ref(Q)
    S = (rnd(Q).double() @ rnd(P).double().T).float()
    if c["block_dict"] is not None:
        for b, q in enumerate(c["queries"]):
            S[b, [pos[p] for p in c["block_dict"][q]]] = -1e6
    v, o = torch.sort(S, dim=1, descending=True, stable=True)
    return v[:, :k].numpy(), o[:, :k].numpy()
