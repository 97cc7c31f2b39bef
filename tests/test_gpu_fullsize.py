"""Parity at the REAL shapes of BASELINE.json's configs, through the C ABI, against the fp32 device
oracle (oracle.score_topk_ref_device: stock torch fp32 products of the bf16-rounded operands with TF32
off, float64 under additive priors, running top-k, ties -> lowest id) under the north_star tolerance
rule, for EVERY query row:

* bench.py's exact workload (configs[2]): 8,841,823 x 768, B = 4096, top-100, history mask -- the
  plan with seeding + histogram sharing + CTA pairs + throttle + two waves;
* NQ shape (configs[1]) as ranking() asks for it: 2,681,468 x 768, B = 3,452, k = 1001;
* one 12.5 M-row shard of the 100 M config (configs[4]): k = 1000, B = 256, global ids, packed keys;
* the crossover sweep (configs[3]) at B = 1 / 128 / 512 / 1024;
* D = 768 with N >= 2^18 (seeded) for SET / ADD / cos.

One 12.5 M x 768 bf16 table (19.2 GB) is generated once per module exactly like bench.py generates
its corpus (same per-chunk seeds); the smaller corpora are its prefixes.  Needs a B200."""
import json
import os
import sys

import numpy as np
import pytest
import torch

import cases
from oracle import ccr_oracle as O
from select_oracle import levers

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-2  # north_star: scores within 1e-2 relative of the fp32 reference for bf16 inputs
N_SHARD, N_MARCO, N_NQ, DIM = 12_500_000, 8_841_823, 2_681_468, 768


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


@pytest.fixture(scope="module")
def bench():
    sys.path.insert(0, ROOT)
    import bench as bench_mod

    return bench_mod


@pytest.fixture(scope="module")
def big(ccr, bench):
    dev = torch.device("cuda:0")
    table = ccr.EmbeddingTable(N_SHARD, DIM, device=dev)
    bench.build_shard(table, 0, N_SHARD, dev)
    # the table rows are what torch's own rounding of the same generator stream gives (first / last chunk)
    for c in (0, (N_SHARD - 1) // bench.CHUNK):
        g = torch.Generator(device=dev).manual_seed(1000 + c)
        rows = torch.randn((bench.CHUNK, DIM), generator=g, device=dev).to(torch.bfloat16)
        a, b = c * bench.CHUNK, min(N_SHARD, (c + 1) * bench.CHUNK)
        assert torch.equal(table.rows[a:b], rows[: b - a])
    yield table
    del table
    torch.cuda.empty_cache()


def _queries(table, B, seed=7):
    return table.encode_queries(torch.randn((B, DIM), generator=torch.Generator().manual_seed(seed)))


def _check(ccr, table, q, N, k, mask, mode=O.MASK_NONE, id_offset=0, **kw):
    out = ccr.score_topk(q, table.data, k, mask=mask, n_items=N, D=table.ld, id_offset=id_offset, want_f64=True, **kw)
    torch.cuda.synchronize()
    s, i, d = out
    ref_s, ref_i = O.score_topk_ref_device(q, table.data, k, mask=mask.host if mask is not None else None,
                                           mode=mode, n_items=N, id_offset=id_offset)
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=ref_s.numpy(), ref_ids=ref_i.numpy(),
                        rtol=RTOL, atol=1e-4)
    assert not errs, errs[:5]
    # position-exact agreement (identical ids at identical ranks), reported for the record
    return float((i.cpu() == ref_i).float().mean()), (s, i, d), (ref_s, ref_i)


def test_bench_workload_every_row_vs_fp32_oracle(ccr, bench, big):
    """bench.py's step: all 4,096 rows (every pair tile, both waves), exact plan asserted."""
    from ccr_b200 import _lib

    dev = big.device
    B, k = 4096, bench.TOPK
    q = _queries(big, B)
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N_MARCO))
    mask = ccr.SparseMask(indptr, cols, vals, N_MARCO, ccr.MASK_SET, dev)
    plan = _lib.plan_info(B, N_MARCO, DIM, k, mask_nnz=mask.nnz, mask_max_row_nnz=mask.max_row_nnz)
    assert plan["two_cta"] == 1 and plan["seed_items"] > 0 and plan["n_q_tiles"] == 16 and plan["algo"] == 2
    agree, (s, i, d), _ = _check(ccr, big, q, N_MARCO, k, mask, O.MASK_SET)
    assert agree > 0.999, agree
    # no blocked passage in any row (each row has far more than k unblocked items)
    rows_of = np.repeat(np.arange(B), np.diff(indptr))
    hit = (i.cpu().numpy()[rows_of] == cols[:, None].astype(np.int64)).any()
    assert not hit
    # the throttle lead, the single-CTA variant and histogram sharing change scheduling only: same bits
    for env in ({"CCR_LEAD": "4"}, {"CCR_2CTA": "0"}, {"CCR_NO_HIST": "1"}):
        with levers(**env):
            s2, i2, d2 = ccr.score_topk(q, big.data, k, mask=mask, n_items=N_MARCO, D=big.ld, want_f64=True)
        assert torch.equal(i, i2) and torch.equal(d, d2), env


def test_nq_shape_k1001_vs_fp32_oracle(ccr, bench, big):
    B, k = 3452, 1001
    q = _queries(big, B, seed=11)
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N_NQ, seed=5))
    mask = ccr.SparseMask(indptr, cols, vals, N_NQ, ccr.MASK_SET, big.device)
    agree, _, _ = _check(ccr, big, q, N_NQ, k, mask, O.MASK_SET)
    assert agree > 0.995, agree
    agree, _, _ = _check(ccr, big, q[:700], N_NQ, k, None)   # ranking() without a block list
    assert agree > 0.995, agree


def test_c5_shard_k1000_global_ids_and_packed_keys(ccr, bench, big):
    """One rank's share of configs[4]: 12.5 M rows, top-1000, ids offset by the shard's first row; the
    packed exchange keys decode to exactly the float32 scores and global ids."""
    B, k, off = 256, 1000, 25_000_000
    q = _queries(big, B, seed=13)
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N_SHARD, seed=6))
    mask = ccr.SparseMask(indptr, cols, vals, N_SHARD, ccr.MASK_SET, big.device)
    agree, (s, i, d), _ = _check(ccr, big, q, N_SHARD, k, mask, O.MASK_SET, id_offset=off)
    assert agree > 0.995 and int(i.min()) >= off
    s2, i2, keys = ccr.score_topk(q, big.data, k, mask=mask, n_items=N_SHARD, D=big.ld, id_offset=off, want_keys=True)
    assert torch.equal(i, i2) and torch.equal(s, s2)
    ku = keys.cpu().numpy().view(np.uint64)
    o = (ku >> np.uint64(32)).astype(np.uint32)
    dec = np.where(o >> 31, o & 0x7FFFFFFF, ~o).astype(np.uint32).view(np.float32)
    np.testing.assert_array_equal(dec, s.cpu().numpy())
    np.testing.assert_array_equal(0xFFFFFFFF - (ku & np.uint64(0xFFFFFFFF)).astype(np.int64), i.cpu().numpy())
    assert bool((ku[:, 1:] < ku[:, :-1]).all())  # strictly descending keys: the merge's precondition
    # merging the run with itself shifted into G = 3 disjoint-id runs gives back the top-k of the union
    runs = torch.stack([keys, keys - 1, keys - 2])  # ids + 1, + 2 at equal scores: distinct, lower rank
    ms, mi = ccr.merge_topk_keys(runs, k)
    flat = np.sort(runs.cpu().numpy().view(np.uint64).transpose(1, 0, 2).reshape(B, -1), axis=1)[:, ::-1][:, :k]
    np.testing.assert_array_equal(mi.cpu().numpy(), 0xFFFFFFFF - (flat & np.uint64(0xFFFFFFFF)).astype(np.int64))
    mk = ccr.merge_topk_keys(runs, k, packed=True)                       # still packed, for a further exchange
    np.testing.assert_array_equal(mk.cpu().numpy().view(np.uint64), flat)
    us, ui = ccr.engine.unpack_topk_keys(mk)
    assert torch.equal(us, ms) and torch.equal(ui, mi)
    us0, ui0 = ccr.engine.unpack_topk_keys(torch.zeros(3, 5, dtype=torch.int64, device=mk.device))
    assert bool((ui0 == -1).all()) and bool(torch.isinf(us0).all())      # key 0 = padding


@pytest.mark.parametrize("B", [1, 128, 512, 1024])
def test_crossover_sweep_batches_vs_fp32_oracle(ccr, big, B):
    agree, _, _ = _check(ccr, big, _queries(big, B, seed=100 + B), N_MARCO, 100, None)
    assert agree > 0.995, agree


SEEDED_D768 = [
    # B, N, k, mode, sim
    (300, 300_000, 100, O.MASK_SET, "dot"),
    (260, 280_000, 1001, O.MASK_ADD, "dot"),
    (140, 270_000, 10, O.MASK_NONE, "cos"),
]


@pytest.mark.parametrize("B,N,k,mode,sim", SEEDED_D768)
def test_seeded_d768_vs_fp32_oracle(ccr, B, N, k, mode, sim):
    """D = 768 (12 K-blocks per tile) at sizes where seeding and the histograms are on; the oracle gets
    the operands as torch rounds them, not as the ingest kernel wrote them."""
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B + N)
    P = torch.as_tensor(cases.embeddings(N % 1000 + 3, N, DIM, clustered=(sim == "cos")))
    Q = torch.as_tensor(cases.embeddings(N % 1000 + 4, B, DIM, clustered=(sim == "cos")))
    table = ccr.EmbeddingTable.from_tensor(P, device=dev, normalize=(sim == "cos"))
    mask = None
    if mode != O.MASK_NONE:
        rows = [rs.choice(N, size=rs.randint(0, 60), replace=False) for _ in range(B)]
        if mode == O.MASK_SET:
            mask = ccr.SparseMask.from_lists(rows, N, -1e6, ccr.MASK_SET, dev)
        else:
            indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
            cols = np.concatenate([np.sort(r) for r in rows])
            vals = np.where(rs.rand(len(cols)) < 0.5, -1e10, rs.choice([1.0, 1e5], size=len(cols)))
            mask = ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_ADD, dev)
    s, i, d = table.search(Q, k, mask=mask, want_f64=True)
    Pe, Qe = P.to(dev), Q.to(dev)
    if sim == "cos":
        Pe, Qe = O.normalize_rows_ref(Pe), O.normalize_rows_ref(Qe)
    Pe, Qe = Pe.to(torch.bfloat16), Qe.to(torch.bfloat16)
    ref_s, ref_i = O.score_topk_ref_device(Qe, Pe, k, mask=mask.host if mask is not None else None, mode=mode)
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=ref_s.numpy(), ref_ids=ref_i.numpy(), rtol=RTOL,
                        atol=2e-3 if sim == "cos" else 1e-4)
    assert not errs, errs[:3]


def test_short_batch_with_strided_queries_and_additive_priors(ccr):
    """B < 128 on the tensor-core kernel stages the queries in a padded block of pitch D; the mask
    override pass must read that block with ITS pitch even when the caller's q is a column slice of a
    wider tensor (advisor finding, round 1)."""
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(3)
    B, N, D, k = 50, 40_000, 128, 20
    P = torch.as_tensor(cases.embeddings(31, N, D))
    wide = torch.randn((B, D + 64), generator=torch.Generator().manual_seed(2)).to(dev).to(torch.bfloat16)
    q = wide[:, :D]
    assert q.stride(0) == D + 64
    table = ccr.EmbeddingTable.from_tensor(P, device=dev)
    rows = [rs.choice(N, size=30, replace=False) for _ in range(B)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    cols = np.concatenate([np.sort(r) for r in rows])
    vals = rs.choice([1e5, 2e5, -1e10], size=len(cols))
    mask = ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_ADD, dev)
    s, i, d = ccr.score_topk(q, table.data, k, mask=mask, n_items=N, D=D, algo=2, want_f64=True)
    ref_s, ref_i = O.score_topk_ref_device(q.contiguous(), table.rows, k, mask=mask.host, mode=O.MASK_ADD)
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=ref_s.numpy(), ref_ids=ref_i.numpy(), rtol=RTOL,
                        atol=1e-4)
    assert not errs, errs[:3]
    assert float(d.max()) > 1e5  # the positive priors decide the top of every row


def test_device_mask_column_shard_equals_host(ccr):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(9)
    B, N = 3000, 1_000_000
    rows = [np.unique(rs.randint(0, N, size=rs.randint(0, 70))) for _ in range(B)]
    mask = ccr.SparseMask.from_lists(rows, N, -1e6, ccr.MASK_SET, dev)
    for lo, hi in [(0, N), (125_000, 250_000), (999_990, N), (5, 5)]:
        h = mask.column_shard(lo, hi)
        g = mask.column_shard_device(lo, hi)
        ip = g.indptr.cpu().numpy()
        np.testing.assert_array_equal(ip, h.host[0])
        n = int(ip[-1])
        np.testing.assert_array_equal(g.cols.cpu().numpy()[:n], h.host[1])
        np.testing.assert_array_equal(g.vals.cpu().numpy()[:n], h.host[2])
        assert g.nnz >= n and g.max_row_nnz >= h.max_row_nnz


def test_bench_dump_outputs_are_the_timed_step(ccr, bench, tmp_path, monkeypatch, capsys):
    """`bench.py --dump-outputs` writes the bits of the timed resident step: a direct search over the
    same seeded table, queries and history mask gives them again.  `--steps` sets how many searches the
    timed loops issue (counted at the table, next to the warm-up ones)."""
    N, B, k, steps, warmup = 300_000, 256, 100, 3, 2
    calls = []
    search = ccr.EmbeddingTable.search
    monkeypatch.setattr(ccr.EmbeddingTable, "search",
                        lambda self, *a, **kw: calls.append(kw.get("encoded", False)) or search(self, *a, **kw))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", str(steps), "--warmup", str(warmup), "--n-items", str(N),
                                      "--batch", str(B), "--no-cpu-baseline", "--no-library-baseline",
                                      "--dump-outputs", str(tmp_path)])
    bench.run_ours(bench.parse())
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == steps
    assert calls.count(True) == warmup + steps              # resident: warm-up + timed
    assert calls.count(False) == max(1, warmup // 2) + steps  # e2e from host buffers: warm-up + timed
    monkeypatch.setattr(ccr.EmbeddingTable, "search", search)
    s, i = np.load(tmp_path / "scores.npy"), np.load(tmp_path / "ids.npy")
    assert s.dtype == np.float32 and i.dtype == np.float64 and s.shape == i.shape == (B, k)
    dev = torch.device("cuda:0")
    table = ccr.EmbeddingTable(N, DIM, device=dev)
    bench.build_shard(table, 0, N, dev)
    q = table.encode_queries(torch.randn((B, DIM), generator=torch.Generator().manual_seed(7)))
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N))
    mask = ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_SET, dev)
    s2, i2 = table.search(q, k, mask=mask, encoded=True)
    np.testing.assert_array_equal(s, s2.cpu().numpy())
    np.testing.assert_array_equal(i, i2.cpu().numpy().astype(np.float64))
