"""fp16 embedding tables (CCR_FLAG_F16) on the device: oracle parity of every kernel path, the bench
workload, the reference's own GPU goldens, al_0_rank's step, ingest numerics and the API.  Needs a B200."""
import io
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
import f16_ref
import select_oracle as SO
from oracle import ccr_oracle as O
from select_oracle import lever, levers  # noqa: F401  (fixture)
from test_gpu_parity import CASES, SEEDED_CASES, _mask  # the same shapes as the bf16 parity tests

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-4  # a hundredth of the bf16 rule: only fp32 accumulation order separates kernel and oracle
F16 = torch.float16


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


@pytest.mark.parametrize("algo", [1, 2])
@pytest.mark.parametrize("B,N,D,k,mode,sim", CASES)
def test_f16_score_topk_matches_oracle(ccr, algo, B, N, D, k, mode, sim):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B * 7 + N)
    P = cases.embeddings(N + 1, N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(N + 2, B, D, clustered=(sim == "cos"))
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"), dtype=F16)
    assert table.dtype == F16 and table.data.dtype == F16
    mask = _mask(rs, B, N, mode, dev, ccr) if mode != O.MASK_NONE else None
    q = table.encode_queries(torch.as_tensor(Q))
    s, i, d = table.search(q, k, mask=mask, algo=algo, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    full = f16_ref.full_scores_ref_f16(Q, P, mask=mask.host if mask else None, mode=mode, sim=sim).numpy()
    live = np.abs(f16_ref.full_scores_ref_f16(Q, P, sim=sim).numpy()).max()
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), full_scores=full, rtol=RTOL, atol=RTOL * float(live))
    assert not errs, errs[:5]
    np.testing.assert_allclose(s.cpu().numpy(), d.cpu().numpy().astype(np.float32), rtol=1e-6)
    errs = SO.check_kernel(algo, s, i, d, q, table.data, table.ld, k, mask, n_items=N)
    assert not errs, errs


@pytest.mark.parametrize("B,N,D,k,mode,sim,two", SEEDED_CASES)
def test_f16_seeded_pair_throttle_paths_match_oracle(ccr, B, N, D, k, mode, sim, two, lever):
    lever(CCR_2CTA=two, CCR_NO_HIST=None)
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B + k)
    P = cases.embeddings(B * 7 + k, N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(B * 11 + k, B, D, clustered=(sim == "cos"))
    P[rs.randint(0, N, size=2000)] = P[rs.randint(0, N, size=2000)]  # some exact ties
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"), dtype=F16)
    mask = _mask(rs, B, N, mode, dev, ccr) if mode != O.MASK_NONE else None
    q = table.encode_queries(torch.as_tensor(Q))
    s, i, d = table.search(q, k, mask=mask, algo=2, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    rs_, ri_ = f16_ref.score_topk_ref_f16(Q, P, k, mask=mask.host if mask else None, mode=mode, sim=sim)
    plain = np.abs(rs_.numpy())
    live = float(plain[plain < 1e4].max())  # largest score without a prior / block value
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=rs_.numpy(), ref_ids=ri_.numpy(), rtol=RTOL,
                        atol=RTOL * live)
    assert not errs, errs[:3]
    errs = SO.check_kernel(2, s, i, d, q, table.data, table.ld, k, mask, n_items=N)
    assert not errs, errs
    # histogram sharing changes scheduling only
    lever(CCR_NO_HIST="1")
    s0, i0, d0 = table.search(q, k, mask=mask, algo=2, want_f64=True, encoded=True)
    assert torch.equal(i, i0) and torch.equal(d.view(torch.int64), d0.view(torch.int64))


def test_f16_bench_workload_every_row(ccr):
    """bench.py's step (8,841,823 x 768, B = 4096, top-100, history mask) on an fp16 table generated like
    bench.build_shard: same plan as bf16, every row against the fp32 device oracle of the fp16 operands."""
    from ccr_b200 import _lib

    sys.path.insert(0, ROOT)
    import bench

    dev = torch.device("cuda:0")
    N, D, B, k = 8_841_823, 768, 4096, bench.TOPK
    table = ccr.EmbeddingTable(N, D, device=dev, dtype=F16)
    bench.build_shard(table, 0, N, dev)
    assert len(table) == N
    g = torch.Generator(device=dev).manual_seed(1000)
    assert torch.equal(table.rows[: bench.CHUNK], torch.randn((bench.CHUNK, D), generator=g, device=dev).half())
    q = table.encode_queries(torch.randn((B, D), generator=torch.Generator().manual_seed(7)))
    assert q.dtype == F16
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N))
    mask = ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_SET, dev)
    kw = dict(mask_nnz=mask.nnz, mask_max_row_nnz=mask.max_row_nnz)
    plan = _lib.plan_info(B, N, D, k, flags=_lib.FLAG_F16, **kw)
    assert plan == _lib.plan_info(B, N, D, k, **kw)
    assert plan["two_cta"] == 1 and plan["seed_items"] > 0 and plan["n_q_tiles"] == 16 and plan["algo"] == 2
    s, i, d = ccr.score_topk(q, table.data, k, mask=mask, n_items=N, D=table.ld, want_f64=True)
    torch.cuda.synchronize()
    ref_s, ref_i = O.score_topk_ref_device(q, table.data, k, mask=mask.host, mode=O.MASK_SET, n_items=N)
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=ref_s.numpy(), ref_ids=ref_i.numpy(),
                        rtol=RTOL, atol=1e-3)
    assert not errs, errs[:5]
    agree = float((i.cpu() == ref_i).float().mean())
    print(f"fp16 bench workload: position-exact {agree:.5f}")
    assert agree >= 0.999, agree
    rows_of = np.repeat(np.arange(B), np.diff(indptr))
    assert not (i.cpu().numpy()[rows_of] == cols[:, None].astype(np.int64)).any()  # no blocked id
    for env in ({"CCR_LEAD": "4"}, {"CCR_2CTA": "0"}, {"CCR_NO_HIST": "1"}):
        with levers(**env):
            s2, i2, d2 = ccr.score_topk(q, table.data, k, mask=mask, n_items=N, D=table.ld, want_f64=True)
        assert torch.equal(i, i2) and torch.equal(d, d2), env
    del table
    torch.cuda.empty_cache()


def _ranking_arrays(prof, c):
    pos = {pid: i for i, pid in enumerate(c["corpus"].keys())}
    qids = list(c["queries"].keys())
    order = np.array([[pos[p] for p in prof[q].keys()] for q in qids])
    scores = np.array([list(prof[q].values()) for q in qids], dtype=np.float32)
    return scores, order


@pytest.mark.parametrize("name", list(cases.CUDA_RANKING_CASES))
def test_f16_ranking_vs_reference_cuda_golden(ccr, name, golden_dir, monkeypatch):
    """ranking(table_dtype=fp16) against the reference's REAL GPU ranking (unmodified ms_marco_eval.ranking
    on a B200 under autocast): the same ranking up to accumulation order, and closer than the bf16 table."""
    g = np.load(os.path.join(golden_dir, f"ranking_cuda_autocast_{name}.npz"))
    c = cases.ranking_case(name)
    monkeypatch.setenv("CCREC_SIM_TYPE", c["sim_type"])
    got = {}
    for label, dt in (("fp16", F16), ("bf16", torch.bfloat16)):
        prof = ccr.ranking(c["corpus"], c["queries"], cases.TextTable(c["table"]), c["batch_size"], c["block_dict"],
                           table_dtype=dt)
        assert list(prof.keys()) == list(c["queries"].keys())
        scores, order = _ranking_arrays(prof, c)
        assert order.shape == g["order"].shape and scores.dtype == np.float32
        got[label] = f16_ref.golden_agreement(scores, order, g["scores"], g["order"])
    print(f"{name}: score-equal / tie-aware / ordered top-2  fp16 {got['fp16']}  bf16 {got['bf16']}")
    eq, tie, top2 = got["fp16"]
    assert eq >= 0.99 and tie >= 0.995 and top2 == 1.0, got["fp16"]
    assert eq > got["bf16"][0] and tie > got["bf16"][1], got


def test_f16_al0_rank_step(ccr, tmp_path, monkeypatch):
    """al_0_rank.py's step on fp16 tables: request CSVs byte-identical to the oracle's restatement of the
    profile it produced, and MRR@1 at least that of the bf16 table."""
    import pandas as pd

    monkeypatch.setenv("CCREC_SIM_TYPE", "dot")
    monkeypatch.setenv("CCREC_DISPLAY_LENGTH", "250")
    c = cases.ranking_case("dot_n1500")
    qids = list(c["queries"])
    bm25 = {q: {p: 1.0 / (r + 1) for r, p in enumerate(list(c["corpus"])[i:i + 50])} for i, q in enumerate(qids)}
    splits = [qids[0::2], qids[1::2]]
    want = O.ranking_ref(c["corpus"], c["queries"], cases.TextTable(c["table"]), c["batch_size"], None, sim_type="dot")
    qrels = {q: {next(iter(want[q])): 1} for q in qids}
    mrr = {}
    for label, dt in (("fp16", F16), ("bf16", torch.bfloat16)):
        out = tmp_path / label
        prof, mrr[label], orig, perm = ccr.al_rank.rank_step(
            c["corpus"], c["queries"], qrels, cases.TextTable(c["table"]), str(out), 3, bm25, splits, n_repeats=2,
            repeat_seed=5, batch_size=c["batch_size"], table_dtype=dt)
        wd = out / "data_iteration_3"
        assert torch.load(wd / "ranking_profile.pt") == prof
        header, rows, permuted, track = O.al0_requests_ref(prof, bm25, c["corpus"], c["queries"], splits, 3, 2, 2, 5)
        buf = io.StringIO()
        pd.DataFrame(permuted, columns=header).to_csv(buf, index=False)
        assert open(wd / "request_perm.csv", "rb").read() == buf.getvalue().encode()
        assert torch.load(wd / "id_track.pt") == track
    print("MRR", mrr)
    assert mrr["fp16"]["MRR@1"] >= mrr["bf16"]["MRR@1"], mrr


def test_f16_ingest_numerics(ccr):
    from ccr_b200 import engine

    dev = torch.device("cuda:0")
    rs = np.random.RandomState(1)
    n, D = 300, 61  # ld = 64: three padding columns
    x = (rs.standard_normal((n, D)) * np.exp(rs.uniform(-20, 11, size=(n, D)))).astype(np.float32)
    x[0, :8] = [65504.0, -65504.0, 65519.0, 6e-8, -3e-8, 1e-5, 0.0, -0.0]  # max, round-down edge, subnormals
    src = torch.as_tensor(x).clamp(-65519, 65519)  # 65519 still rounds to 65504
    dst = torch.full((n, 64), float("nan"), dtype=F16, device=dev)
    ovf = torch.zeros(1, dtype=torch.int32, device=dev)
    engine.ingest_rows(src.to(dev), dst, normalize=False, overflow=ovf)
    assert int(ovf.item()) == 0
    want = src.to(F16)
    assert torch.equal(dst[:, :D].cpu().view(torch.int16), want.view(torch.int16))  # bit for bit, -0 included
    assert bool((dst[:, D:] == 0).all())
    # L2-normalised: within one fp16 ulp of F.normalize(x).half()
    y = torch.as_tensor(rs.standard_normal((n, D)).astype(np.float32))
    engine.ingest_rows(y.to(dev), dst, normalize=True)
    ref = torch.nn.functional.normalize(y, p=2, dim=1).half()
    ulp = torch.as_tensor(np.spacing(np.abs(ref.numpy()).astype(np.float16)).astype(np.float32))
    assert bool(((dst[:, :D].cpu().float() - ref.float()).abs() <= ulp).all())
    # overflow: the batch is refused and the table keeps its length
    t = ccr.EmbeddingTable(4, D, device=dev, dtype=F16)
    t.append(src[:3])
    bad = torch.zeros(2, D)
    bad[1, 5] = 70000.0
    with pytest.raises(ValueError, match="1 value"):
        t.append(bad)
    assert len(t) == 3
    with pytest.raises(ValueError, match="overflow"):
        t.encode_queries(bad)
    # fp16 sources are copied, bf16 sources widened and rounded once
    h = torch.as_tensor(rs.standard_normal((5, D)).astype(np.float32)).half()
    b = torch.as_tensor(rs.standard_normal((5, D)).astype(np.float32)).to(torch.bfloat16)
    t.append(h).append(b)
    assert len(t) == 13
    assert torch.equal(t.rows[3:8, :D].cpu().view(torch.int16), h.view(torch.int16))
    assert torch.equal(t.rows[8:13, :D].cpu().view(torch.int16), b.float().half().view(torch.int16))
    tn = ccr.EmbeddingTable(0, D, device=dev, normalize=True, dtype=F16).append(h)
    ref = torch.nn.functional.normalize(h.float(), p=2, dim=1).half()
    assert float((tn.rows[:, :D].cpu().float() - ref.float()).abs().max()) <= 2 ** -11


@pytest.mark.parametrize("B,N,D", [(300, 5000, 768), (130, 9001, 200), (1, 1_100_000, 64), (5, 100, 768),
                                   (40, 900, 64)])
def test_f16_dense_scores_match_fp32_product(ccr, B, N, D):
    """ccr_score_dense_f16 on both paths (>= 2^20 scores: tcgen05 store tiles; fewer: CUDA cores)."""
    dev = torch.device("cuda:0")
    P = torch.as_tensor(cases.embeddings(N % 97, N, D))
    Q = torch.as_tensor(cases.embeddings(N % 89, B, D))
    table = ccr.EmbeddingTable.from_tensor(P, device=dev, dtype=F16)
    got = table.dense_scores(Q)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = table.encode_queries(Q).float()[:, :D] @ table.rows.float()[:, :D].T
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    assert got.shape == (B, N) and got.dtype == torch.float32
    torch.testing.assert_close(got, want, rtol=1e-4, atol=2e-3)


def test_f16_api_checks_and_persistence(ccr, tmp_path):
    from ccr_b200 import engine

    dev = torch.device("cuda:0")
    P = torch.randn(3000, 64)
    t16 = ccr.EmbeddingTable.from_tensor(P, device=dev, dtype=F16)
    t16b = ccr.EmbeddingTable.from_tensor(P, device=dev)
    q16, qb = t16.encode_queries(P[:4]), t16b.encode_queries(P[:4])
    for q, items in ((q16, t16b.data), (qb, t16.data)):
        with pytest.raises(TypeError):
            engine.score_topk(q, items, 5, n_items=3000)
        with pytest.raises(TypeError):
            engine.score_dense(q, items, n_items=3000)
    s, i = engine.score_topk(q16, t16.data, 5, n_items=3000)
    assert bool((i[:, 0] == torch.arange(4, device=dev)).all())  # each query is its own best row
    path = str(tmp_path / "t.pt")
    t16.save(path)
    back = ccr.EmbeddingTable.load(path, device=dev)
    assert back.dtype == F16 and len(back) == len(t16)
    assert torch.equal(back.rows.view(torch.int16), t16.rows.view(torch.int16))
    # a file written without the dtype key (before fp16 tables existed) loads as bf16
    blob = torch.load(path)
    blob.pop("dtype")
    blob["rows"] = t16b.rows.cpu()
    torch.save(blob, path)
    old = ccr.EmbeddingTable.load(path, device=dev)
    assert old.dtype == torch.bfloat16 and torch.equal(old.rows, t16b.rows)


@pytest.mark.parametrize("world", [2])
def test_f16_sharded_index_equals_one_table(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    port = 29800 + world + os.getpid() % 100
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_f16_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-4000:]
    assert r.returncode == 0, tail
    assert r.stdout.count("f16_equal_single_table=True") == 5 * world, tail
