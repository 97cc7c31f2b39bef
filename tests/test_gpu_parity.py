"""Parity of the CUDA path (through the C ABI) against the CPU oracle.  Needs a B200."""
import os

import numpy as np
import pytest
import scipy.sparse as sps
import torch

import cases
import select_oracle as SO
from oracle import ccr_oracle as O
from select_oracle import lever  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

RTOL = 1e-2  # north_star: scores within 1e-2 relative of the fp32 reference for bf16 inputs


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


def _mask(rs, B, N, mode, dev, ccr, max_h=40):
    rows = [rs.choice(N, size=min(N, rs.randint(0, max_h)), replace=False) for _ in range(B)]
    if mode == O.MASK_SET:
        return ccr.SparseMask.from_lists(rows, N, -1e6, ccr.MASK_SET, dev)
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    cols = np.concatenate([np.sort(r) for r in rows]) if B else np.zeros(0)
    vals = np.where(rs.rand(len(cols)) < 0.5, -1e10, rs.choice([1.0, 1e5], size=len(cols)))
    return ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_ADD, dev)


CASES = [
    # B, N, D, k, mode, sim
    (1, 257, 64, 5, O.MASK_NONE, "dot"),
    (3, 1000, 768, 100, O.MASK_SET, "dot"),
    (8, 5000, 768, 1001, O.MASK_NONE, "dot"),
    (17, 3000, 128, 7, O.MASK_ADD, "dot"),
    (130, 4000, 768, 100, O.MASK_SET, "cos"),
    (64, 20000, 200, 10, O.MASK_ADD, "dot"),
    (300, 30000, 768, 100, O.MASK_NONE, "dot"),
    (129, 2500, 768, 1001, O.MASK_SET, "dot"),
    (5, 40, 768, 40, O.MASK_SET, "dot"),  # k == N: blocked items come last
]


@pytest.mark.parametrize("algo", [1, 2])
@pytest.mark.parametrize("B,N,D,k,mode,sim", CASES)
def test_score_topk_matches_oracle(ccr, algo, B, N, D, k, mode, sim):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B * 7 + N)
    P = cases.embeddings(N + 1, N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(N + 2, B, D, clustered=(sim == "cos"))
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"))
    mask = _mask(rs, B, N, mode, dev, ccr) if mode != O.MASK_NONE else None
    q = table.encode_queries(torch.as_tensor(Q))
    s, i, d = table.search(q, k, mask=mask, algo=algo, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    full = O.full_scores_ref(Q, P, mask=mask.host if mask else None, mode=mode, sim=sim).numpy()
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), full_scores=full, rtol=RTOL)
    assert not errs, errs[:5]
    np.testing.assert_allclose(s.cpu().numpy(), d.cpu().numpy().astype(np.float32), rtol=1e-6)
    errs = SO.check_kernel(algo, s, i, d, q, table.data, table.ld, k, mask, n_items=N)
    assert not errs, errs


@pytest.mark.parametrize("algo", [1, 2])
def test_exact_ties_break_by_lowest_id(ccr, algo):
    dev = torch.device("cuda:0")
    N, D, B, k = 3000, 64, 9, 50
    P = np.zeros((N, D), dtype=np.float32)
    P[:, 0] = np.repeat(np.arange(N // 10), 10)[::-1]  # runs of 10 identical scores
    Q = np.zeros((B, D), dtype=np.float32)
    Q[:, 0] = 1.0
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev)
    s, i = table.search(torch.as_tensor(Q), k, algo=algo)
    rs_, ri_ = O.score_topk_ref(Q, P, k)
    np.testing.assert_array_equal(i.cpu().numpy(), ri_.numpy())
    np.testing.assert_array_equal(s.cpu().numpy(), rs_.numpy())


@pytest.mark.parametrize("algo", [1, 2])
def test_all_zero_scores(ccr, algo):
    dev = torch.device("cuda:0")
    table = ccr.EmbeddingTable.from_tensor(torch.zeros(5000, 64), device=dev)
    s, i = table.search(torch.zeros(4, 64), 300, algo=algo)
    np.testing.assert_array_equal(i.cpu().numpy(), np.tile(np.arange(300), (4, 1)))
    assert float(s.abs().max()) == 0.0


def test_k_out_of_range_raises_like_torch(ccr):
    dev = torch.device("cuda:0")
    table = ccr.EmbeddingTable.from_tensor(torch.randn(10, 64), device=dev)
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        table.search(torch.randn(2, 64), 11)
    with pytest.raises(ValueError):
        table.search(torch.randn(2, 64), 5000)


def test_empty_query_batch(ccr):
    dev = torch.device("cuda:0")
    table = ccr.EmbeddingTable.from_tensor(torch.randn(100, 64), device=dev)
    s, i = table.search(torch.zeros(0, 64), 5)
    assert s.shape == (0, 5) and i.shape == (0, 5)


@pytest.mark.parametrize("name", list(cases.RANKING_CASES))
def test_ranking_dropin_vs_golden(ccr, name, golden_dir, monkeypatch):
    """ccr_b200.ranking on the inputs the goldens were made from (outputs of the unmodified
    reference): same keys/order up to bf16 near-ties, scores within tolerance."""
    g = np.load(os.path.join(golden_dir, f"ranking_{name}.npz"))
    c = cases.ranking_case(name)
    monkeypatch.setenv("CCREC_SIM_TYPE", c["sim_type"])
    prof = ccr.ranking(c["corpus"], c["queries"], cases.TextTable(c["table"]), c["batch_size"], c["block_dict"])
    pos = {pid: i for i, pid in enumerate(c["corpus"].keys())}
    qids = list(c["queries"].keys())
    assert list(prof.keys()) == qids
    order = np.array([[pos[p] for p in prof[q].keys()] for q in qids])
    scores = np.array([list(prof[q].values()) for q in qids])
    assert order.shape == g["order"].shape
    # the golden is the reference's fp32 arithmetic on UNROUNDED inputs; the device table is
    # bf16, so the tolerance is 1e-2 relative to the scale of the live (unblocked) scores
    live = g["scores"][g["scores"] > -1e6]
    errs = O.check_topk(scores, order, ref_scores=g["scores"], ref_ids=g["order"], rtol=RTOL,
                        atol=RTOL * float(np.abs(live).max()))
    assert not errs, errs[:5]
    # blocked passages carry exactly -1e6
    if c["block_dict"] is not None:
        for b, q in enumerate(qids):
            blocked = {pos[p] for p in c["block_dict"][q]}
            got_blocked = order[b][scores[b] == -1e6]
            assert set(got_blocked) <= blocked


@pytest.mark.parametrize("name", list(cases.CUDA_RANKING_CASES))
def test_ranking_dropin_vs_reference_cuda_golden(ccr, name, golden_dir, monkeypatch):
    """The drop-in against the reference's REAL GPU path: goldens = unmodified ms_marco_eval.ranking on a
    B200 under torch.cuda.amp.autocast() (fp16 tensor-core scores, SURVEY.md section 8c(3)).  north_star
    rule: scores within 1e-2 relative, id sets equal up to near-ties at the k-th score."""
    g = np.load(os.path.join(golden_dir, f"ranking_cuda_autocast_{name}.npz"))
    c = cases.ranking_case(name)
    monkeypatch.setenv("CCREC_SIM_TYPE", c["sim_type"])
    prof = ccr.ranking(c["corpus"], c["queries"], cases.TextTable(c["table"]), c["batch_size"], c["block_dict"])
    pos = {pid: i for i, pid in enumerate(c["corpus"].keys())}
    qids = list(c["queries"].keys())
    assert list(prof.keys()) == qids
    order = np.array([[pos[p] for p in prof[q].keys()] for q in qids])
    scores = np.array([list(prof[q].values()) for q in qids])
    assert order.shape == g["order"].shape
    live = g["scores"][g["scores"] > -1e6]
    errs = O.check_topk(scores, order, ref_scores=g["scores"], ref_ids=g["order"], rtol=RTOL,
                        atol=RTOL * float(np.abs(live).max()))
    assert not errs, errs[:5]
    # the pairs the labelling requests are built from (al_0_rank.py:172): same top-2 set in most rows
    # (fp16 vs bf16 rounding may swap near-ties)
    same_top2 = np.mean([set(order[b, :2]) == set(g["order"][b, :2]) for b in range(len(qids))])
    assert same_top2 >= 0.8, same_top2


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_assign_topk_dropin_vs_golden(ccr, name, golden_dir):
    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = ccr.LazyDenseMatrix(c["U"]) @ ccr.LazyDenseMatrix(c["V"]).T
    if c["prior"] is not None:
        S = S + c["prior"]
    csr = ccr._assign_topk(S, c["k"], device="cpu")
    assert csr.shape == tuple(g["shape"])
    np.testing.assert_array_equal(csr.indptr, g["indptr"])
    np.testing.assert_array_equal(csr.data, g["data"])
    got = csr.indices.reshape(len(c["U"]), c["k"])
    dense = O.lazy_score_dense_ref(c["U"], c["V"], c["prior"]).numpy()
    sc = np.take_along_axis(dense, got, 1)
    errs = O.check_topk(sc, got, full_scores=dense, rtol=RTOL)
    assert not errs, errs[:5]
    # at these sizes bf16 rounding rarely flips a rank: most rows match the reference exactly
    assert (got == g["indices"]).all(axis=1).mean() > 0.7


def test_evaluate_item_rec_metrics(ccr, golden_dir):
    name = "mask_prior_k1"
    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = ccr.LazyDenseMatrix(c["U"]) @ ccr.LazyDenseMatrix(c["V"]).T + c["prior"]
    ref_assigned = sps.csr_matrix((g["data"], g["indices"].ravel(), g["indptr"]), shape=tuple(g["shape"]))
    m = ccr.evaluate_item_rec(ref_assigned, S, c["k"])
    want = dict(zip(g["metric_names"].tolist(), g["metric_values"].tolist()))
    for key in ("prec", "recs/user", "item_cov", "user_cov", "recall"):
        assert abs(m[key] - want[key]) < 0.06, (key, m[key], want[key])
    assert abs(m["obj_mean"] - want["obj_mean"]) / abs(want["obj_mean"]) < RTOL


@pytest.mark.parametrize("G,B,k", [(4, 37, 20), (8, 48, 1000), (2, 5, 2048), (8, 3, 2048)])
def test_merge_topk_matches_oracle(ccr, G, B, k):
    """(8, 3, 2048) exceeds the shared-memory staging of the merge and takes the global-memory path."""
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(3)
    sc = np.sort(rs.standard_normal((G, B, k)), axis=2)[:, :, ::-1].copy()
    sc[1, :, k // 2:] = sc[0, :, k // 2:]  # cross-run ties
    ids = rs.permutation(G * B * k).reshape(G, B, k).astype(np.int64)
    ids[G - 1, :, 3 * k // 4:] = -1  # padding
    s, i, d = ccr.merge_topk(torch.as_tensor(sc).to(dev), torch.as_tensor(ids).to(dev), k)
    for b in range(B):
        ent = [(-sc[g_, b, j], ids[g_, b, j]) for g_ in range(G) for j in range(k) if ids[g_, b, j] >= 0]
        ent.sort()
        np.testing.assert_array_equal(i[b].cpu().numpy(), [e[1] for e in ent[:k]])
        np.testing.assert_array_equal(d[b].cpu().numpy(), [-e[0] for e in ent[:k]])


def test_property_full_size_sample(ccr):
    """Size-independent properties at a large shape: order, uniqueness, threshold consistency,
    and agreement between the two kernels (SIMT vs tcgen05) on the same rows."""
    dev = torch.device("cuda:0")
    N, D, k = 1_000_003, 768, 100
    g = torch.Generator(device=dev).manual_seed(7)
    items = torch.randn((N, D), generator=g, device=dev).to(torch.bfloat16)
    q = torch.randn((136, D), generator=g, device=dev).to(torch.bfloat16)
    s2, i2 = ccr.score_topk(q, items, k, algo=2)
    s1, i1 = ccr.score_topk(q[:8], items, k, algo=1)
    assert bool((s2[:, 1:] <= s2[:, :-1]).all())
    assert all(len(set(r.tolist())) == k for r in i2.cpu())
    torch.testing.assert_close(s1, s2[:8], rtol=1e-4, atol=1e-3)
    assert (i1 == i2[:8]).float().mean().item() > 0.98
    # every returned score equals the recomputed dot product
    re = (q[:4].float() @ items[i2[:4].reshape(-1)].float().T)
    re = torch.stack([re[r, r * k:(r + 1) * k] for r in range(4)])
    torch.testing.assert_close(re, s2[:4], rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_argsort_dropin_vs_golden(ccr, name, golden_dir):
    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = ccr.LazyDenseMatrix(c["U"]) @ ccr.LazyDenseMatrix(c["V"]).T
    if c["prior"] is not None:
        S = S + c["prior"]
    r, col = ccr._argsort(S, tie_breaker=0)
    assert len(r) == S.shape[0] * S.shape[1]
    dense = O.lazy_score_dense_ref(c["U"], c["V"], c["prior"]).numpy().astype(np.float64)
    got = dense[r, col]
    scale = np.abs(dense[np.abs(dense) < 1e4]).max()
    # descending up to the bf16 tolerance, and the head agrees with the reference's own order
    assert np.all(np.diff(got) <= RTOL * scale + RTOL * np.abs(got[1:]))
    agree = np.mean((r[:64] == g["argsort_rows"]) & (col[:64] == g["argsort_cols"]))
    assert agree > 0.5


def test_mrr_matches_manual(ccr):
    order = np.array([[3, 1, 2], [0, 2, 1], [2, 0, 1]])
    corpus_ids, qids = ["a", "b", "c", "d"], ["q0", "q1", "q2"]
    qrels = {"q0": {"b": 1}, "q1": {"d": 1}, "q2": {"c": 1, "a": 0}}
    m = ccr.mrr_at_k(order, corpus_ids, qids, qrels, k_values=(1, 3))
    assert m == {"MRR@1": round(1 / 3, 5), "MRR@3": round((0.5 + 0 + 1) / 3, 5)}


def test_empty_shard_pads(ccr):
    dev = torch.device("cuda:0")
    q = torch.randn(5, 64, device=dev).to(torch.bfloat16)
    items = torch.zeros(0, 64, device=dev, dtype=torch.bfloat16)
    s, i = ccr.score_topk(q, items, 7, allow_short=True)
    assert bool((i == -1).all()) and bool(torch.isinf(s).all())
    items = torch.randn(3, 64, device=dev).to(torch.bfloat16)
    s, i = ccr.score_topk(q, items, 7, allow_short=True, id_offset=100)
    assert bool((i[:, :3] >= 100).all()) and bool((i[:, 3:] == -1).all())


def test_full_corpus_properties(ccr):
    """BASELINE size (8,841,823 x 768), B=300, k=100 with history mask: order, uniqueness, no
    blocked id returned, every returned score equals the recomputed dot product, and the k-th
    score dominates a random sample of non-returned items."""
    dev = torch.device("cuda:0")
    N, D, B, k = 8_841_823, 768, 300, 100
    items = torch.empty((N, D), dtype=torch.bfloat16, device=dev)
    g = torch.Generator(device=dev).manual_seed(11)
    for s0 in range(0, N, 1 << 20):
        e = min(N, s0 + (1 << 20))
        items[s0:e] = torch.randn((e - s0, D), generator=g, device=dev).to(torch.bfloat16)
    q = torch.randn((B, D), generator=g, device=dev).to(torch.bfloat16)
    rs = np.random.RandomState(3)
    rows = [np.unique(rs.randint(0, N, size=rs.randint(0, 65))) for _ in range(B)]
    # make the mask bite: block each row's true best item as well
    s0_, i0_ = ccr.score_topk(q, items, 1)
    rows = [np.unique(np.append(r, int(i0_[b, 0]))) for b, r in enumerate(rows)]
    mask = ccr.SparseMask.from_lists(rows, N, -1e6, ccr.MASK_SET, dev)
    s, i = ccr.score_topk(q, items, k, mask=mask)
    assert bool((s[:, 1:] <= s[:, :-1]).all())
    assert all(len(set(r.tolist())) == k for r in i.cpu())
    for b in range(0, B, 37):
        assert not set(i[b].tolist()) & set(rows[b].tolist())
        re = (q[b].float() @ items[i[b]].float().T)
        torch.testing.assert_close(re, s[b], rtol=1e-4, atol=1e-3)
        probe = torch.as_tensor(rs.randint(0, N, size=20000), device=dev)
        probe = probe[~torch.isin(probe, i[b]) & ~torch.isin(probe, torch.as_tensor(rows[b], device=dev))]
        assert float((q[b].float() @ items[probe].float().T).max()) <= float(s[b, -1]) + 1e-3


# ---- shapes large enough (N >= 2^18) for the threshold-seeding pre-pass and the per-row histogram
# ---- sharing to be active, checked against the CPU oracle under the north_star tolerance rule
SEEDED_CASES = [
    # B, N, D, k, mode, sim, two_cta
    (200, 300_000, 128, 10, O.MASK_NONE, "dot", "1"),
    (300, 300_000, 128, 1001, O.MASK_SET, "dot", "0"),
    (256, 270_000, 64, 100, O.MASK_ADD, "dot", "1"),
    (130, 400_000, 64, 2048, O.MASK_NONE, "cos", "0"),
    (5, 300_000, 128, 100, O.MASK_SET, "dot", "0"),
    # default policy (None): several query tiles per item split -> CTA pairs + bounded-drift throttle
    (2304, 280_000, 64, 50, O.MASK_NONE, "dot", None),
    (1100, 300_000, 64, 100, O.MASK_SET, "dot", None),   # 9 tiles: odd -> single CTAs, two waves
    (4200, 270_000, 64, 10, O.MASK_ADD, "dot", None),    # 33 tiles -> 17 pair tiles, padded rows
]


@pytest.mark.parametrize("B,N,D,k,mode,sim,two", SEEDED_CASES)
def test_seeded_histogram_path_matches_oracle(ccr, B, N, D, k, mode, sim, two, lever):
    lever(CCR_2CTA=two, CCR_NO_HIST=None)
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B + k)
    P = cases.embeddings(B * 7 + k, N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(B * 11 + k, B, D, clustered=(sim == "cos"))
    P[rs.randint(0, N, size=2000)] = P[rs.randint(0, N, size=2000)]  # some exact ties
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"))
    mask = _mask(rs, B, N, mode, dev, ccr) if mode != O.MASK_NONE else None
    q = table.encode_queries(torch.as_tensor(Q))
    s, i, d = table.search(q, k, mask=mask, algo=2, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    rs_, ri_ = O.score_topk_ref(Q, P, k, mask=mask.host if mask else None, mode=mode, sim=sim)
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=rs_.numpy(), ref_ids=ri_.numpy(), rtol=RTOL,
                        atol=2e-3 if sim == "cos" else 1e-4)
    assert not errs, errs[:3]
    errs = SO.check_kernel(2, s, i, d, q, table.data, table.ld, k, mask, n_items=N)
    assert not errs, errs
    # and the histogram sharing must not change a single bit of the result
    lever(CCR_NO_HIST="1")
    s0, i0, d0 = table.search(q, k, mask=mask, algo=2, want_f64=True, encoded=True)
    assert torch.equal(i, i0) and torch.equal(d.view(torch.int64), d0.view(torch.int64))


def test_seeded_path_degenerate_scores(ccr):
    """All-zero table at a seeded size: every score ties, positions 0..k-1 must come back; and a
    table whose rows are all the same vector (one distinct score per query)."""
    dev = torch.device("cuda:0")
    N, D, k = 300_000, 64, 7
    q = torch.randn(150, D, device=dev).to(torch.bfloat16)
    s, i = ccr.score_topk(q, torch.zeros(N, D, device=dev, dtype=torch.bfloat16), k, algo=2)
    assert bool((i == torch.arange(k, device=dev)).all()) and float(s.abs().max()) == 0.0
    row = torch.randn(1, D, device=dev).to(torch.bfloat16)
    s, i = ccr.score_topk(q, row.expand(N, D).contiguous(), k, algo=2)
    assert bool((i == torch.arange(k, device=dev)).all())
    torch.testing.assert_close(s[:, 0], (q.float() @ row.float().T)[:, 0], rtol=1e-4, atol=1e-3)


def test_al0_rank_step_end_to_end(ccr, tmp_path, monkeypatch):
    """al_0_rank.py:107-218 through ccr_b200.al_rank.rank_step: dense retrieval on the device,
    ranking_profile.pt written and reused, MRR, and request CSVs byte-identical to the oracle's
    restatement applied to the same profile."""
    import io

    import pandas as pd

    monkeypatch.setenv("CCREC_SIM_TYPE", "dot")
    monkeypatch.setenv("CCREC_DISPLAY_LENGTH", "250")
    c = cases.ranking_case("dot_n1500")
    table = cases.TextTable(c["table"])
    qids = list(c["queries"])
    bm25 = {q: {p: 1.0 / (r + 1) for r, p in enumerate(list(c["corpus"])[i:i + 50])} for i, q in enumerate(qids)}
    splits = [qids[0::2], qids[1::2]]
    want = O.ranking_ref(c["corpus"], c["queries"], cases.TextTable(c["table"]), c["batch_size"], None, sim_type="dot")
    qrels = {q: {next(iter(want[q])): 1} for q in qids}  # the oracle's best passage is the relevant one
    prof, mrr, orig, perm = ccr.al_rank.rank_step(c["corpus"], c["queries"], qrels, table, str(tmp_path), 3, bm25,
                                                  splits, n_repeats=2, repeat_seed=5, batch_size=c["batch_size"])
    assert mrr["MRR@1"] > 0.8 and mrr["MRR@5"] > 0.99  # bf16 table: a near-tie at rank 1 may swap
    assert len(orig) == len(splits[1]) and len(perm) == 2 * len(orig)
    wd = tmp_path / "data_iteration_3"
    assert torch.load(wd / "ranking_profile.pt") == prof
    header, rows, permuted, track = O.al0_requests_ref(prof, bm25, c["corpus"], c["queries"], splits, 3, 2, 2, 5)
    buf = io.StringIO()
    pd.DataFrame(permuted, columns=header).to_csv(buf, index=False)
    assert open(wd / "request_perm.csv", "rb").read() == buf.getvalue().encode()
    assert torch.load(wd / "id_track.pt") == track
    calls = table.calls
    ccr.al_rank.rank_step(c["corpus"], c["queries"], qrels, table, str(tmp_path), 3, bm25, splits, 2, 5)
    assert table.calls == calls  # cached profile: the encoder is not called again


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_assign_topk_on_materialised_matrix_is_bit_exact(ccr, name, golden_dir):
    """The reference's unmodified ``transform`` hands ``_assign_topk`` a dense host matrix (+ prior):
    same fp32 matrix in -> the reference's own indices out, exactly (no bf16 anywhere)."""
    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    dense = O.lazy_score_dense_ref(c["U"], c["V"], None).numpy()  # fp32 U @ V.T as the reference builds it
    S = ccr.LazyDenseMatrix(dense)
    if c["prior"] is not None:
        S = S + c["prior"]
    csr = ccr._assign_topk(S, c["k"])
    idx = csr.indices.copy()  # scipy comparisons below sort csr.indices in place
    np.testing.assert_array_equal(idx.reshape(len(c["U"]), c["k"]), g["indices"])
    np.testing.assert_array_equal(csr.indptr, g["indptr"])
    m = ccr.evaluate_item_rec((csr > 0).astype(np.float64), S, c["k"])
    want = dict(zip(g["metric_names"].tolist(), g["metric_values"].tolist()))
    for key, v in want.items():
        # obj_mean: the reference sums fp32 scores in fp32 when no float64 prior is added
        assert abs(m[key] - v) <= 1e-5 * max(1.0, abs(v)), (key, m[key], v)
    csr2 = ccr._assign_topk(dense if c["prior"] is None else S, c["k"])  # plain ndarray input too
    np.testing.assert_array_equal(csr2.indices, idx)


@pytest.mark.parametrize("B,N,k,mode", [(7, 5000, 100, O.MASK_NONE), (300, 20000, 1001, O.MASK_ADD),
                                        (2, 300_000, 10, O.MASK_SET), (40, 37, 37, O.MASK_ADD),
                                        (1100, 3000, 5, O.MASK_NONE)])
def test_topk_dense_abi_matches_float64_sort(ccr, B, N, k, mode):
    """ccr_topk_dense_f32 (materialised score matrix + sparse prior) against the reference's
    arithmetic: float32 scores, promoted to float64 where a prior is added / assigned, stable
    descending order.  Heavy exact ties (scores drawn from 50 distinct values in some rows)."""
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B + N + k)
    dense = rs.standard_normal((B, N)).astype(np.float32)
    dense[::3] = rs.randint(0, 50, size=dense[::3].shape).astype(np.float32)  # tie-heavy rows
    mask = _mask(rs, B, N, mode, dev, ccr, max_h=min(N, 30)) if mode != O.MASK_NONE else None
    s, i, d = ccr.topk_dense(torch.as_tensor(dense).to(dev), k, mask=mask)
    full = torch.as_tensor(dense).double()
    if mask is not None:
        indptr, cols, vals = mask.host
        for r in range(B):
            c = torch.as_tensor(cols[indptr[r]:indptr[r + 1]].astype(np.int64))
            v = torch.as_tensor(vals[indptr[r]:indptr[r + 1]])
            full[r, c] = v if mode == O.MASK_SET else full[r, c] + v
    want_v, want_i = torch.sort(full, dim=1, descending=True, stable=True)
    np.testing.assert_array_equal(i.cpu().numpy(), want_i[:, :k].numpy())
    np.testing.assert_array_equal(d.cpu().numpy(), want_v[:, :k].numpy())
    np.testing.assert_array_equal(s.cpu().numpy(), want_v[:, :k].float().numpy())
    with pytest.raises(RuntimeError, match="out of range"):
        ccr.topk_dense(torch.zeros(2, 3, device=dev), 4)


@pytest.mark.parametrize("sim", ["dot", "cos"])
def test_transform_scores_topk_vs_reference_matrix(ccr, sim):
    """bbpr.py:528-550 replaced by the lazy factor pair: top-k (+ prior) through the fused kernel
    against the reference's dense matrix path under the tolerance rule."""
    rs = np.random.RandomState(8)
    all_emb = cases.embeddings(77, 900, 64, clustered=(sim == "cos"))
    i_to_ptr, j_to_ptr = rs.randint(0, 900, size=33), rs.permutation(900)[:700]
    prior = sps.csr_matrix((np.full(33, -1e10), (np.arange(33), rs.randint(0, 700, size=33))), shape=(33, 700))
    S = ccr.transform_scores(all_emb, i_to_ptr, j_to_ptr, sim_type=sim) + prior
    got = ccr._assign_topk(S, 10).indices.reshape(33, 10)
    dense = O.transform_scores_ref(all_emb, i_to_ptr, j_to_ptr, 256, sim).double().numpy() + prior.toarray()
    got_scores = np.take_along_axis(dense, got, 1)
    errs = O.check_topk(got_scores, got, full_scores=dense, rtol=RTOL, atol=2e-3 if sim == "cos" else 1e-4)
    assert not errs, errs[:3]


@pytest.mark.parametrize("B,N,mode", [(7, 300, O.MASK_NONE), (300, 5001, O.MASK_ADD), (64, 40_000, O.MASK_SET),
                                      (1, 1, O.MASK_NONE), (1500, 7000, O.MASK_ADD)])
def test_argsort_abi_matches_stable_float64_sort(ccr, B, N, mode):
    """ccr_argsort_scores_f32 (whole-matrix LSD radix sort; rime_lite _argsort's device core) against a
    stable descending float64 sort of the same matrix with the priors merged as the reference promotes
    them; tie-heavy rows included.  Bit-exact (rows, cols)."""
    from ccr_b200 import engine

    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B + N)
    dense = rs.standard_normal((B, N)).astype(np.float32)
    dense[::3] = rs.randint(-20, 20, size=dense[::3].shape).astype(np.float32)  # ties, negatives, zeros
    mask = _mask(rs, B, N, mode, dev, ccr, max_h=min(N, 30)) if mode != O.MASK_NONE else None
    rows, cols = engine.argsort_scores(torch.as_tensor(dense).to(dev), mask)
    full = torch.as_tensor(dense).double()
    if mask is not None:
        indptr, mc, mv = mask.host
        for r in range(B):
            c = torch.as_tensor(mc[indptr[r]:indptr[r + 1]].astype(np.int64))
            v = torch.as_tensor(mv[indptr[r]:indptr[r + 1]])
            full[r, c] = v if mode == O.MASK_SET else full[r, c] + v
    want = torch.sort(full.reshape(-1), descending=True, stable=True).indices.numpy()
    np.testing.assert_array_equal(rows.cpu().numpy() * N + cols.cpu().numpy(), want)


@pytest.mark.parametrize("B,N,D", [(300, 5000, 768), (130, 9001, 200), (1, 1_100_000, 64), (5, 100, 768)])
def test_dense_score_tile_matches_fp32_product(ccr, B, N, D):
    """ccr_score_dense_f32: tiles of >= 2^20 scores run on the TMA + tcgen05 pipeline with a store
    epilogue (ragged last tile, row pitch not a multiple of 4), smaller ones on the CUDA-core kernel;
    both against torch's fp32 product of the bf16-rounded operands."""
    dev = torch.device("cuda:0")
    P = torch.as_tensor(cases.embeddings(N % 97, N, D))
    Q = torch.as_tensor(cases.embeddings(N % 89, B, D))
    table = ccr.EmbeddingTable.from_tensor(P, device=dev)
    got = table.dense_scores(Q)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = table.encode_queries(Q).float()[:, :D] @ table.rows.float()[:, :D].T
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    assert got.shape == (B, N)
    torch.testing.assert_close(got, want, rtol=1e-4, atol=2e-3)


def test_lazy_matmul_as_tensor_on_cuda_uses_the_device_kernel(ccr):
    rs = np.random.RandomState(4)
    U, V = rs.standard_normal((40, 64)).astype(np.float32), rs.standard_normal((900, 64)).astype(np.float32)
    S = ccr.LazyDenseMatrix(U) @ ccr.LazyDenseMatrix(V).T
    got = S.as_tensor("cuda")
    assert got.is_cuda and got.dtype == torch.float32 and tuple(got.shape) == (40, 900)
    want = O.bf16_round(torch.as_tensor(U)) @ O.bf16_round(torch.as_tensor(V)).T
    torch.testing.assert_close(got.cpu(), want, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(S.as_tensor("cpu"), torch.as_tensor(U) @ torch.as_tensor(V).T)  # host path unchanged


def test_first_hit_rank_and_mrr_denominator(ccr):
    from ccr_b200 import engine

    dev = torch.device("cuda:0")
    rs = np.random.RandomState(5)
    B, k, N = 500, 100, 5000
    ids = np.stack([rs.permutation(N)[:k] for _ in range(B)]).astype(np.int64)
    rel = [np.unique(rs.randint(0, N, size=rs.randint(0, 6))) for _ in range(B)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rel])]).astype(np.int64)
    got = engine.first_hit_rank(torch.as_tensor(ids).to(dev), indptr, np.concatenate(rel)).cpu().numpy()
    want = np.zeros(B, dtype=np.int32)
    for b in range(B):
        hit = np.nonzero(np.isin(ids[b], rel[b]))[0]
        want[b] = hit[0] + 1 if hit.size else 0
    np.testing.assert_array_equal(got, want)
    # BEIR divides by len(qrels), not by the number of ranked queries
    corpus_ids = [f"p{i}" for i in range(N)]
    qids = [f"q{b}" for b in range(B)]
    qrels = {q: {corpus_ids[c]: 1 for c in rel[b]} for b, q in enumerate(qids)}
    qrels["never_ranked"] = {"p0": 1}
    m = ccr.mrr_at_k(ids, corpus_ids, qids, qrels, k_values=(1, 10, 100))
    for kk in (1, 10, 100):
        ok = (want > 0) & (want <= kk)
        assert m[f"MRR@{kk}"] == round(float(np.sum(1.0 / want[ok])) / (B + 1), 5)
