"""The host side of the dense and BM25 top-k plan matrices (tests/test_gpu_select_dense_bm25.py), no GPU needed.

* The plan mirrors in select_oracle.py equal the library's plans: their totals are what the size queries return
  (the plans are exported nowhere else), over a grid of shapes.  Without a device the library plans for 148
  SMs, the mirrors' default; with one it uses the device's count, so that test is skipped there.
* The BM25 accumulation oracle on synthetic postings is bit-identical to the reference's BM25 on a small sklearn
  corpus when its impacts are computed in the header's operation order: the synthetic-index cases check
  against the reference's arithmetic.
* The dense oracle's NaN rule and mask merge, on a hand-written row."""
import itertools

import numpy as np
import pytest
import torch

import select_oracle as SO
from ccr_b200 import _lib
from oracle import ccr_oracle as O

no_device = pytest.mark.skipif(torch.cuda.is_available(), reason="the library plans for the device's SM count")

SHAPES = [(B, N, k) for B, N, k in itertools.product([1, 2, 7, 40, 300, 2000, 4096, 65535],
                                                      [1, 37, 511, 4096, 20_011, 300_000, 4_300_000],
                                                      [1, 10, 1001, 2048]) if k <= N]


@no_device
def test_dense_plan_mirror_matches_the_size_query():
    L = _lib.lib()
    for (B, N, k), (nnz, h) in itertools.product(SHAPES, [(0, 0), (5000, 0), (5000, 48), (64 * 7, 64), (1, 300)]):
        if k + h > _lib.MAX_K:
            continue
        plan = SO.dense_plan(B, N, k, nnz, h)
        assert L.ccr_topk_dense_workspace_bytes(B, N, k, nnz, h) == plan["total"], (B, N, k, nnz, h)
        cols = SO.dense_split_cols(plan, N)
        assert cols[0][0] == 0 and cols[-1][1] == N and all(a[1] == b[0] for a, b in zip(cols, cols[1:]))


@no_device
def test_bm25_plan_mirror_matches_the_size_query():
    L = _lib.lib()
    for B, N, k in SHAPES:
        warp, block = SO.bm25_plan(B, N, k, True), SO.bm25_plan(B, N, k, False)
        assert L.ccr_bm25_topk_workspace_bytes(B, N, k) == max(warp["total"], block["total"]), (B, N, k)
        assert L.ccr_bm25_topk_workspace_bytes(B, N, k) == SO.bm25_workspace(B, N, k)
        assert warp["streams"] <= SO.FIN_MAX_STREAMS and block["streams"] <= SO.FIN_MAX_STREAMS
        for plan in (warp, block):
            docs = SO.bm25_stream_docs(plan, N)
            assert docs[0][0] == 0 and docs[-1][1] == N


def test_plan_mirror_branches_at_148_sms():
    """The branches the GPU matrix pins, for the B200's 148 SMs (the GPU cases recompute them for the device)."""
    assert SO.dense_plan(1, 4_300_000, 2048)["S"] == 1024
    assert SO.dense_plan(7, 300_000, 1001, 7 * 64, 64)["S"] == 74
    assert SO.dense_plan(2000, 4096, 2000, 1, 48)["S"] == 1
    assert SO.dense_plan(40, 20_000, 100, 800, 300)["S"] == 5
    assert SO.dense_plan(64, 40_000, 100)["S"] == 10
    assert SO.dense_finalize_entries(SO.dense_plan(2000, 4096, 2000, 1, 48), 4096, 2048, 48) == (4096, 4096)
    cap = SO.bm25_plan(1, 1_000_000, 2048, True)
    assert (cap["S"], cap["streams"]) == (128, 1024)
    assert SO.bm25_plan(4, 300_000, 1001, True)["per"] == SO.BMW_MINI
    assert SO.bm25_plan(600, 300_000, 1001, True)["S"] == 1
    assert SO.bm25_plan(2, 2_100_000, 1001, False)["S"] == 370
    assert SO.bm25_workspace(65535, 600, 10) > 2 << 30


def _bm25_index(ref):
    """(post_indptr, post_docs, post_val) of a fitted BM25Ref, impacts in the header's operation order."""
    csc = ref.csc
    norm = ref.k1 * (1 - ref.b + ref.b * ref.doc_len / ref.avdl)
    idf = ref.vectorizer._tfidf.idf_ - 1.0
    term = np.repeat(np.arange(csc.shape[1]), np.diff(csc.indptr))
    val = SO.bm25_post_val(csc.data, idf[term], norm[csc.indices], ref.k1)
    return csc.indptr.astype(np.int64), csc.indices.astype(np.int32), val


def test_bm25_accumulation_oracle_is_the_reference():
    rs = np.random.RandomState(3)
    vocab = [f"w{i}" for i in range(400)]
    p = 1.0 / np.arange(1, 401)
    p /= p.sum()
    corpus = [" ".join(rs.choice(vocab, size=rs.randint(3, 60), p=p)) for _ in range(3000)]
    queries = [" ".join(rs.choice(vocab, size=rs.randint(1, 40), p=p)) for _ in range(50)] + ["zzunseen", "",
                                                                                          " ".join(vocab[::7])]
    ref = O.BM25Ref(b=0.75, k1=1.2).fit(corpus)
    ip, docs, val = _bm25_index(ref)
    q = ref.counts(queries).tocsr()
    q.sort_indices()
    assert np.diff(q.indptr).max() > SO.BMW_MAX_TERMS
    got = SO.bm25_scores(ip, docs, val, q.indptr, q.indices, len(corpus)).numpy()
    for b, text in enumerate(queries):
        want = ref.transform(text)
        assert np.array_equal(got[b].view(np.int64), want.view(np.int64)), b


def test_dense_oracle_nan_rule_and_mask_merge():
    """SET replaces the value, ADD adds it to double(score); NaN never ranks (a row with fewer than k other
    values ends in (-inf, -1)); ties go to the lower id; -0.0 ranks just below +0.0; -inf ranks."""
    nan, inf = float("nan"), float("inf")
    row = np.array([1.0, nan, 3.0, 3.0, -inf, 0.0, -0.0, nan, 2.0, 5.0], dtype=np.float32)
    full = torch.as_tensor(row).double()[None].clone()
    # mask: col 2 SET -1e30, col 9 ADD 0.5 (5.5), col 1 ADD 1.0 on a NaN cell (NaN: never ranks)
    full[0, 2] = -1e30
    full[0, 9] = float(row[9]) + 0.5
    full[0, 1] = float(row[1]) + 1.0
    v, i = SO.exact_topk(full, 10, drop_nan=True)
    assert i[0].tolist() == [9, 3, 8, 0, 5, 6, 2, 4, -1, -1]
    want = [5.5, 3.0, 2.0, 1.0, 0.0, -0.0, -1e30, -inf, -inf, -inf]
    assert v[0].numpy().view(np.int64).tolist() == np.array(want).view(np.int64).tolist()
    v, i = SO.exact_topk(full, 5, drop_nan=True)
    assert i[0].tolist() == [9, 3, 8, 0, 5]
    # without NaN the two paths of exact_topk agree
    clean = torch.nan_to_num(full, nan=7.0)
    a, b = SO.exact_topk(clean, 10, drop_nan=True), SO.exact_topk(clean, 10)
    assert torch.equal(a[1], b[1]) and torch.equal(a[0].view(torch.int64), b[0].view(torch.int64))
