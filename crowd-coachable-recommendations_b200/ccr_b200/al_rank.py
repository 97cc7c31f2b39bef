"""Step 0 of the human-in-the-loop cycle with the same inputs and outputs as
scripts/al_0_rank.py: ``ranking_profile.pt`` (cached per step, :111-127), MRR@{1,5,10,100}
(:130-133), 4-candidate labelling tasks = dense top-2 + first unseen BM25 hit + random fill
(:165-182), ``id_track.pt`` / ``request_orig.csv`` / ``request_perm.csv`` (:196-218).

The script itself is module-level code that is not importable at the reference's HEAD (it imports
``load_corpus`` / ``load_query`` that do not exist, SURVEY.md §0) and drags in the encoder; here
the same step is a function of already-loaded inputs.  Only the ``ranking(...)`` call runs on the
device (ccr_b200.ranking); everything after it is host bookkeeping whose byte-for-byte output is
pinned by tests/golden/al0_*.npz (produced by executing the reference's own statements).

Random draws follow the reference exactly: candidates use ``RandomState(STEP)`` with one
``choice(len(corpus))`` per attempt, the display order uses ``RandomState(REPEAT_SEED)`` with one
``permutation(4)`` per emitted row.
"""
from __future__ import annotations

import os
import re

import numpy as np
import torch

HEADER = ["query", "passage-1", "passage-2", "passage-3", "passage-4", "qid", "pid-1", "pid-2", "pid-3", "pid-4"]
IMAGE_HEADER = ["img-q", "img-1", "img-2", "img-3", "img-4"]
_KEEP = re.compile(r"[^a-zA-Z0-9 ,:.;?$!()&\[\]]")


def filter_string(text, display_length=None):
    """Characters the MTurk layout may show, cut to CCREC_DISPLAY_LENGTH (al_0_rank.py:142-144)."""
    if display_length is None:
        display_length = int(os.environ["CCREC_DISPLAY_LENGTH"])
    return _KEEP.sub("", text)[:display_length]


def mrr_from_profile(qrels, ranking_profile, k_values=(1, 5, 10, 100)):
    """MRR@k as al_0_rank.py:130-133 obtains it from BEIR (``EvaluateRetrieval.evaluate_custom(qrels,
    results, k_values, metric="mrr")`` -- third party, unvendored and unpinned by the reference;
    its published algorithm: per query the results are ordered by score, the reciprocal rank of the
    first hit with qrels score > 0 inside the top k is summed, the sum is divided by ``len(qrels)``
    and rounded to 5 digits).  A ``RankingProfile`` (what ``ccr_b200.ranking`` returns) is scored from
    its [Q, k] position array by the device first-hit scan; a plain dict takes the per-query loop."""
    from .ranking import RankingProfile, mrr_at_k

    if isinstance(ranking_profile, RankingProfile) and ranking_profile.order.ndim == 2 and len(ranking_profile):
        for qid in ranking_profile.queries_ids:
            qrels[qid]  # BEIR indexes qrels[query_id] for every result: KeyError for an unknown query
        return mrr_at_k(ranking_profile.order[:, : max(k_values)], ranking_profile.corpus_ids.tolist(),
                        ranking_profile.queries_ids, qrels, k_values)
    k_max = max(k_values)
    sums = {k: 0.0 for k in k_values}
    for qid, scored in ranking_profile.items():
        relevant = {pid for pid, rel in qrels.get(qid, {}).items() if rel > 0}
        if not relevant:
            continue
        top = sorted(scored.items(), key=lambda kv: kv[1], reverse=True)[:k_max]
        first = next((r for r, (pid, _) in enumerate(top) if pid in relevant), None)
        if first is not None:
            for k in k_values:
                if first < k:
                    sums[k] += 1.0 / (first + 1)
    n = max(1, len(qrels))
    return {f"MRR@{k}": round(sums[k] / n, 5) for k in k_values}


def select_candidates(ranks, ranks_bm25, corpus_keys, rng):
    """Dense top-2, then the best BM25 passage not among them, then random corpus passages until
    there are four distinct ones (al_0_rank.py:169-182)."""
    cands = list(ranks[:2])
    for pid in ranks_bm25:  # normally adds exactly one; more only if the dense list is shorter than 2
        if len(cands) >= 3:
            break
        if pid not in cands:
            cands.append(pid)
    while len(cands) < 4:
        pid = corpus_keys[rng.choice(len(corpus_keys))]
        if pid not in cands:
            cands.append(pid)
    return cands


class _Draws:
    """The reference's ``RandomState(STEP).choice(len(corpus))`` stream, drawn in blocks: a bulk
    ``randint(0, n, size=m)`` yields exactly the values of m scalar ``choice(n)`` calls (legacy
    MT19937 stream, checked in tests/test_al_rank_cpu.py), at a fraction of the call overhead."""

    def __init__(self, rng, n, block=4096):
        self.rng, self.n, self.block = rng, n, block
        self.buf = np.zeros(0, dtype=np.int64)
        self.ptr = 0

    def take(self, m):
        """The next m draws (consumed)."""
        have = len(self.buf) - self.ptr
        if have < m:
            more = self.rng.randint(0, self.n, size=max(self.block, m - have))
            self.buf = np.concatenate([self.buf[self.ptr:], more])
            self.ptr = 0
        out = self.buf[self.ptr : self.ptr + m]
        self.ptr += m
        return out

    def give_back(self, m):
        self.ptr -= m


def _fill_fourth(cand_pos, draws):
    """For queries that hold exactly three candidates (corpus positions [Q, 3]): the fourth is the first
    draw of the stream that is not one of the three -- queries in order, each consuming draws until one
    is accepted (al_0_rank.py:178-182).  Vectorised: a run of queries takes one draw each until the
    first rejection, which is resolved sequentially."""
    Q = len(cand_pos)
    fourth = np.empty(Q, dtype=np.int64)
    i = 0
    while i < Q:
        m = Q - i
        d = draws.take(m)
        clash = (d[:, None] == cand_pos[i : i + m]).any(axis=1)
        j = int(np.argmax(clash)) if clash.any() else m
        fourth[i : i + j] = d[:j]
        draws.give_back(m - j)          # only j draws were really consumed
        i += j
        if j < m:                       # query i rejected its draw: keep drawing for it alone
            while True:
                dd = int(draws.take(1)[0])
                if dd not in cand_pos[i]:
                    fourth[i] = dd
                    i += 1
                    break
    return fourth


def build_requests(ranking_profile, ranking_profile_bm25, corpus, queries, split_qids, step, landing_image=None):
    """-> (header, rows, id_track) for the queries of this step's split, in ranking_profile order."""
    rng = np.random.RandomState(step)
    corpus_keys = list(corpus.keys())
    wanted = split_qids if isinstance(split_qids, (set, frozenset)) else set(np.asarray(split_qids).tolist())
    header = HEADER + (IMAGE_HEADER if landing_image is not None else [])
    top_ids = getattr(ranking_profile, "top_ids", None)
    qids = [qid for qid in ranking_profile if qid in wanted]
    # dense top-2, then the best BM25 passage not among them (al_0_rank.py:169-177)
    all_cands = []
    for qid in qids:
        cands = top_ids(qid, 2) if top_ids is not None else list(ranking_profile[qid].keys())[:2]
        for pid in ranking_profile_bm25[qid].keys():
            if len(cands) >= 3:
                break
            if pid not in cands:
                cands.append(pid)
        all_cands.append(cands)
    # random corpus passages until there are four distinct ones (:178-182), same draw sequence
    draws = _Draws(rng, len(corpus_keys))
    if qids and all(len(c) == 3 for c in all_cands):
        pos = {pid: i for i, pid in enumerate(corpus_keys)}
        cand_pos = np.array([[pos[p] for p in c] for c in all_cands], dtype=np.int64)
        for c, f in zip(all_cands, _fill_fourth(cand_pos, draws)):
            c.append(corpus_keys[f])
    else:  # short dense / BM25 lists: some query needs several random picks -> plain sequential loop
        for c in all_cands:
            while len(c) < 4:
                pid = corpus_keys[int(draws.take(1)[0])]
                if pid not in c:
                    c.append(pid)
    rows, id_track = [], {}
    for qid, cands in zip(qids, all_cands):
        passages = [filter_string(corpus[pid]) for pid in cands]
        row = [queries[qid], *passages, f"q_{qid}", *(f"p_{pid}" for pid in cands)]
        if landing_image is not None:
            row += [landing_image[qid], *(landing_image[pid] for pid in cands)]
        rows.append(row)
        id_track[queries[qid]] = f"q_{qid}"
        id_track.update({text: f"p_{pid}" for pid, text in zip(cands, passages)})
    return header, rows, id_track


def permute_requests(rows, n_repeats, repeat_seed):
    """n_repeats copies of every task with its four passages (and ids, images) shown in an
    independently drawn order (al_0_rank.py:204-215)."""
    rng = np.random.RandomState(repeat_seed)
    out = []
    for _ in range(n_repeats):
        for row in rows:
            order = rng.permutation(4)
            shown = [row[0], *(row[1 + i] for i in order), row[5], *(row[6 + i] for i in order)]
            if len(row) > 10:
                shown += [row[10], *(row[11 + i] for i in order)]
            out.append(shown)
    return out


def write_requests(working_dir, header, rows, id_track, n_repeats, repeat_seed):
    """id_track.pt, request_orig.csv, request_perm.csv exactly as al_0_rank.py:196-218 writes them."""
    import pandas as pd
    import torch

    os.makedirs(working_dir, exist_ok=True)
    torch.save(id_track, os.path.join(working_dir, "id_track.pt"))
    request_orig = pd.DataFrame(rows, columns=header)
    request_orig.to_csv(os.path.join(working_dir, "request_orig.csv"), index=False)
    request_perm = pd.DataFrame(permute_requests(rows, n_repeats, repeat_seed), columns=header)
    request_perm.to_csv(os.path.join(working_dir, "request_perm.csv"), index=False)
    return request_orig, request_perm


def generate_train_data(qids, qrels, ranking_profile, ranking_profile_2, corpus_key_list=(), rng_seed=None):
    """Oracle-labelled training tasks of the notebook loop (scripts/al_oracle_agent.py:134-180): per
    query the dense top-2, then BM25 passages up to four candidates -- or, with ``corpus_key_list``, up
    to three plus one random corpus passage as attention check (``RandomState(rng_seed)``, one
    ``choice`` per attempt) -- shuffled with the global ``random`` module exactly once per query like
    the reference; a candidate listed in ``qrels[qid]`` becomes the positive (the last one if several),
    the others negatives; queries without a labelled candidate are skipped in the attention-check
    variant and keep the shuffled head as positive otherwise."""
    import random

    rng = np.random.RandomState(rng_seed)
    train_data = {}
    for qid in qids:
        pids = list(ranking_profile[qid].keys())[:2]
        for pid in ranking_profile_2[qid].keys():
            if len(pids) == 4:
                break
            if pid not in pids:
                pids.append(pid)
        if len(corpus_key_list):
            pids = pids[:3]
            while len(pids) < 4:
                pid = corpus_key_list[rng.choice(len(corpus_key_list))]
                if pid not in pids:
                    pids.append(pid)
        random.shuffle(pids)
        labelled = [pid for pid in pids if pid in qrels[qid]]
        if labelled:
            train_data[qid] = {"pos_pid": [labelled[-1]], "neg_pid": [pid for pid in pids if pid not in qrels[qid]]}
        elif not len(corpus_key_list):
            train_data[qid] = {"pos_pid": pids[:1], "neg_pid": pids[1:]}
    return train_data


def rank_step(corpus, queries, qrels, embedding_func, results_dir, step, ranking_profile_bm25, qids_split,
              n_repeats=3, repeat_seed=42, number_of_qid_split_batch=None, block_dict=None, landing_image=None,
              batch_size=512, device="cuda", table_dtype=torch.bfloat16, exact=False):
    """al_0_rank.py:107-218 as a function: reuse or compute ``data_iteration_{step}/ranking_profile.pt``
    (the dense retrieval runs through ccr_b200.ranking on the device, on tables of ``table_dtype``:
    bf16 by default, fp16 to rank on the reference's own autocast operand format), report MRR, write
    the labelling requests.  Returns (ranking_profile, mrr, request_orig, request_perm)."""

    from .ranking import ranking

    working_dir = os.path.join(results_dir, f"data_iteration_{step}")
    os.makedirs(working_dir, exist_ok=True)
    profile_path = os.path.join(working_dir, "ranking_profile.pt")
    if os.path.isfile(profile_path):
        ranking_profile = torch.load(profile_path)
    else:
        ranking_profile = ranking(corpus, queries, embedding_func, batch_size, block_dict, device=device,
                                  table_dtype=table_dtype, exact=exact)
        # the reference's file format is the plain dict (loadable with torch.load's weights-only default)
        torch.save(ranking_profile.to_dict() if hasattr(ranking_profile, "to_dict") else ranking_profile, profile_path)
    mrr = mrr_from_profile(qrels, ranking_profile, [1, 5, 10, 100])
    for name, value in mrr.items():
        print(name, ":", value)
    split = qids_split[step % (number_of_qid_split_batch or len(qids_split))]
    header, rows, id_track = build_requests(ranking_profile, ranking_profile_bm25, corpus, queries, split, step,
                                            landing_image)
    request_orig, request_perm = write_requests(working_dir, header, rows, id_track, n_repeats, repeat_seed)
    return ranking_profile, mrr, request_orig, request_perm
