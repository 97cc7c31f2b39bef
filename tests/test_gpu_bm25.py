"""BM25 on the device (ccr_b200.BM25 / ranking_bm25 through the C ABI) against the reference's
golden outputs and the CPU oracle.  Needs a B200.

Bar: the float64 score vectors are BIT-identical to scripts/bm_25.py (same operations in the same
order); the float32 ranking is identical except inside runs of exactly tied scores, where the
reference's unstable sort leaves the order (and, at the 1001 cut, the membership) unspecified and
this path takes the lowest corpus position.
"""
import os

import numpy as np
import pytest
import torch

import cases
import select_oracle as SO
from ccr_b200 import bm25
from oracle import ccr_oracle as O
from select_oracle import lever  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


def _check_order(order, scores, want_order, want_scores):
    np.testing.assert_array_equal(scores, want_scores)  # float32 values, exactly
    for b in range(len(order)):
        if np.array_equal(order[b], want_order[b]):
            continue
        diff = order[b] != want_order[b]
        for v in np.unique(scores[b][diff]):
            run = scores[b] == v
            cut = np.nonzero(run)[0][-1] == order.shape[1] - 1  # run cut by the top-n slice
            if not cut:
                assert set(order[b][run]) == set(want_order[b][run])
        assert len(set(order[b].tolist())) == order.shape[1]


@pytest.mark.parametrize("name", list(cases.BM25_CASES))
def test_bm25_golden_replay(name, golden_dir, ccr):
    g = np.load(os.path.join(golden_dir, f"bm25_{name}.npz"))
    c = cases.bm25_case(name)
    texts = list(c["corpus"].values())
    qids = list(c["queries"].keys())
    model = ccr.BM25(b=0.75, k1=1.2).fit(texts)
    assert float(model.avdl) == float(g["avdl"])
    for i in range(len(g["dense"])):  # BM25.transform drop-in: float64, bit-identical
        np.testing.assert_array_equal(model.transform(c["queries"][qids[i]]), g["dense"][i])
    dense = model.scores([c["queries"][q] for q in qids[: len(g["dense"])]]).cpu().numpy()
    np.testing.assert_array_equal(dense, g["dense"])
    model16 = ccr.BM25().fit(texts)
    np.testing.assert_array_equal(model16.scores([c["queries"][q] for q in qids[:4]]).cpu().numpy(), g["dense_k16"])
    prof = ccr.ranking_bm25(c["corpus"], c["queries"])
    assert list(prof.keys()) == qids
    pos = {pid: i for i, pid in enumerate(c["corpus"].keys())}
    order = np.array([[pos[p] for p in prof[q].keys()] for q in qids])
    scores = np.array([list(prof[q].values()) for q in qids])
    assert order.shape == g["order"].shape
    _check_order(order, scores, g["order"], g["scores"])


def _synthetic(seed, n, q, vocab, doc_len):
    rs = np.random.RandomState(seed)
    corpus = [cases._zipf_text(rs, vocab, rs.randint(3, doc_len)) for _ in range(n)]
    queries = [cases._zipf_text(rs, vocab, rs.randint(1, 14)) for _ in range(q)]
    queries[0] = corpus[7]                       # a whole passage as query (many terms)
    queries[1] = "zzunseen"                      # no vocabulary term: all scores 0
    queries[2] = " ".join(f"w{vocab - 1 - i}" for i in range(6))  # rare terms only: mostly zero scores
    return corpus, queries


@pytest.fixture(params=["auto", "blockwide"])
def bm25_kernel(request, lever):
    """auto: queries of <= 32 distinct terms take the warp-private kernel, longer ones the block-wide
    kernel (the batches below hold both kinds); blockwide: everything on the block-wide kernel."""
    lever(CCR_BM25_BLOCKWIDE="1" if request.param == "blockwide" else None)
    return request.param


@pytest.mark.parametrize("n,q,k", [(40000, 40, 1001), (150000, 300, 100), (9000, 700, 10), (20000, 4100, 100)])
def test_bm25_topk_vs_oracle(n, q, k, ccr, bm25_kernel):
    """Every row: the exact top k (float32 ranking, ties to the lowest position) of the model's own float64
    scores; sampled rows also against the reference's arithmetic.  4,100 queries cross BM25.topk's 4096-query
    chunks; every 97th and the second-to-last are three passages long (> 32 distinct terms), so both chunks
    split into a warp-kernel call and a block-wide call whose rows are put back in place."""
    corpus, queries = _synthetic(41 + k, n, q, vocab=20000, doc_len=60)
    if q > bm25.QUERY_CHUNK:
        for b in list(range(50, q, 97)) + [q - 2]:
            queries[b] = " ".join(corpus[b % n: b % n + 3])
    model = ccr.BM25(b=0.75, k1=1.2).fit(corpus)
    ref = O.BM25Ref(b=0.75, k1=1.2).fit(corpus)
    s, i = model.topk(queries, k)
    if q > bm25.QUERY_CHUNK:
        lengths = np.diff(model.encode_queries(queries)[0])
        for c in range(0, q, bm25.QUERY_CHUNK):
            assert lengths[c: c + bm25.QUERY_CHUNK].max() > bm25.WARP_KERNEL_MAX_TERMS
    want_v, want_i = SO.exact_topk(model.scores(queries).float(), k)
    errs = SO.check_exact(s.cpu().numpy(), i.cpu().numpy(), s.double().cpu().numpy(), want_v.cpu().numpy(),
                          want_i.cpu().numpy())
    assert not errs, errs
    s, i = s.cpu().numpy(), i.cpu().numpy()
    check = range(q) if q <= 64 else list(range(8)) + list(range(8, q, max(1, q // 24)))
    for b in check:
        full = torch.Tensor(ref.transform(queries[b]))
        ws, wi = full.sort(descending=True, stable=True)
        np.testing.assert_array_equal(s[b], ws[:k].numpy())
        np.testing.assert_array_equal(i[b], wi[:k].numpy())  # both: ties -> lowest position
    # every returned score is the document's own score (all rows)
    dense = model.scores(queries[:16])
    got = torch.gather(dense, 1, torch.as_tensor(i[:16]).to(dense.device)).float().cpu().numpy()
    np.testing.assert_array_equal(got, s[:16])


def test_bm25_dense_scores_vs_oracle_many_chunks(ccr):
    """n_docs spanning many 4096-doc accumulator chunks and doc splits; long postings lists."""
    corpus, queries = _synthetic(5, 70000, 12, vocab=500, doc_len=30)
    model = ccr.BM25().fit(corpus)
    ref = O.BM25Ref().fit(corpus)
    dense = model.scores(queries).cpu().numpy()
    for b, text in enumerate(queries):
        np.testing.assert_array_equal(dense[b], ref.transform(text))


def test_bm25_head_rows_bit_identical(ccr):
    """Dense float64 rows for the head terms (hybrid index) change the memory traffic, not a single bit of
    the scores: postings only == default fraction == nearly every term dense, on both kernels (the batch
    holds short queries and a whole passage) with n_docs not a multiple of the 512-doc chunk."""
    corpus, queries = _synthetic(17, 33333, 64, vocab=300, doc_len=40)
    queries.append(" ".join(corpus[i] for i in range(3, 15)))   # a long query: block-wide kernel
    n_terms = [len(set(q.split())) for q in queries]
    assert sum(n <= 32 for n in n_terms) >= 20 and max(n_terms) > 32
    short = [q for q, n in zip(queries, n_terms) if n <= 32]
    model = ccr.BM25(b=0.75, k1=1.2, head_df_fraction=None).fit(corpus)
    assert model.head_terms().size == 0
    want = model.scores(queries).cpu().numpy()          # longest query > 32 terms: block-wide kernel
    want_short = model.scores(short).cpu().numpy()      # warp-private kernel
    ws, wi = model.topk(queries, 1001)                  # short / long queries split between the two
    ref = O.BM25Ref(b=0.75, k1=1.2).fit(corpus)
    np.testing.assert_array_equal(want[3], ref.transform(queries[3]))
    sizes = []
    for frac in (0.25, 0.05, 1e-4):
        model.head_df_fraction = frac
        model._impacts_stale = True
        got = model.scores(queries).cpu().numpy()
        sizes.append(model.head_terms().size)
        assert model._head_rows is not None and model._head_rows.shape[0] == sizes[-1]
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(model.scores(short).cpu().numpy(), want_short)
        s, i = model.topk(queries, 1001)
        assert torch.equal(s, ws) and torch.equal(i, wi)
    assert 0 < sizes[0] <= sizes[1] <= sizes[2] == 64  # capped at HEAD_MAX_TERMS


def test_bm25_edge_cases(ccr):
    corpus, queries = _synthetic(9, 500, 4, vocab=200, doc_len=12)
    model = ccr.BM25().fit(corpus)
    s, i = model.topk([], 5)
    assert s.shape == (0, 5) and i.shape == (0, 5)
    with pytest.raises(RuntimeError, match="out of range"):
        model.topk(queries, 501)
    s, i = model.topk(["zzunseen"], 500)  # k == N, all-zero scores: positions in order
    np.testing.assert_array_equal(i.cpu().numpy()[0], np.arange(500))
    assert float(s.abs().max()) == 0.0
    wide = ccr.BM25().fit([" ".join(f"w{j}" for j in range(r, r + 350)) for r in (0, 350)])
    with pytest.raises(ValueError, match="distinct terms"):
        wide.topk([" ".join(f"w{j}" for j in range(700))], 1)
    s2, i2 = wide.topk([" ".join(f"w{j}" for j in range(500))], 2)  # 500 distinct terms: fine
    assert i2.cpu().numpy().tolist() == [[0, 1]]
    # re-caching other documents (transform(q, X)) keeps the fitted vocabulary / idf / avdl
    other = corpus[:100]
    ref = O.BM25Ref().fit(corpus)
    ref.cache(other)
    np.testing.assert_array_equal(model.transform(queries[3], other), ref.transform(queries[3]))
    assert ccr.ranking_bm25({f"p{j}": t for j, t in enumerate(corpus)}, {}) == {}
