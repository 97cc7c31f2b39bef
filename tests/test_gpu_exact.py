"""Exact fp32 ranking (EmbeddingTable(exact=True), DESIGN.md section 6b) against a float64 oracle.  Needs a B200.

The oracle: the table's stored fp32 rows multiplied in float64, rounded to fp32, the mask applied (SET: the
value, ADD: double(score) + value) and a stable (value descending, id ascending) sort."""
import numpy as np
import pytest
import torch

import cases
from oracle import ccr_oracle as O
from select_oracle import lever, levers  # noqa: F401  (fixture)
from test_gpu_parity import CASES, _mask  # the parity shapes

pytestmark = pytest.mark.gpu

SCANS = {"bf16": torch.bfloat16, "fp16": torch.float16}


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


def _rows32(table, q32):
    return table.data32[: table.n].double().cpu().numpy(), q32.double().cpu().numpy()


def _amb(s64, s32):
    """Items whose float64 sum lies within 2^-40 relative of an fp32 rounding midpoint: the kernel's own
    float64 sum (another order) may round them the other way, by 1 ulp."""
    lo = np.nextafter(s32, np.float32(-np.inf)).astype(np.float64)
    hi = np.nextafter(s32, np.float32(np.inf)).astype(np.float64)
    c = s32.astype(np.float64)
    mid = np.minimum(np.abs(s64 - (lo + c) / 2), np.abs(s64 - (hi + c) / 2))
    return mid <= np.abs(s64) * 2.0 ** -40


def oracle(table, q32, k, mask=None):
    """(values float64 [B,N], ids [B,k] of the exact ranking, ambiguous items [B,N])."""
    P, Q = _rows32(table, q32)
    s64 = Q @ P.T
    s32 = s64.astype(np.float32)
    val = s32.astype(np.float64)
    amb = _amb(s64, s32)
    if mask is not None:
        ip, c, v = mask.host
        for r in range(len(ip) - 1):
            cols = c[ip[r] : ip[r + 1]]
            if mask.mode == O.MASK_SET:
                val[r, cols] = v[ip[r] : ip[r + 1]]
                amb[r, cols] = False
            else:
                val[r, cols] = val[r, cols] + v[ip[r] : ip[r + 1]]
    N = val.shape[1]
    ids = np.stack([np.lexsort((np.arange(N), -val[r]))[:k] for r in range(val.shape[0])]) if len(val) else \
        np.zeros((0, k), dtype=np.int64)
    return val, ids, amb


def compare_rows(val_of, amb_of, oi, s, i, d):
    """Exact agreement with the oracle; the only waiver is an item flagged ambiguous: its value may differ by
    1 fp32 ulp, and a position may hold another item only when the item there or the oracle's is ambiguous.
    val_of(r, ids) / amb_of(r, ids) give the oracle's values / flags of items of row r."""
    for r in range(len(oi)):
        got_amb, ref_amb = amb_of(r, i[r]), amb_of(r, oi[r])
        want = val_of(r, i[r])
        exact_ok = (d[r] == want) | (got_amb & (np.abs(d[r].astype(np.float32).astype(np.float64) - want)
                                                <= np.abs(np.spacing(want.astype(np.float32))).astype(np.float64)))
        assert exact_ok.all(), (r, np.nonzero(~exact_ok)[0][:5], d[r][~exact_ok][:3], want[~exact_ok][:3])
        np.testing.assert_array_equal(s[r], d[r].astype(np.float32))
        pos_ok = (i[r] == oi[r]) | got_amb | ref_amb
        assert pos_ok.all(), (r, np.nonzero(~pos_ok)[0][:5], i[r][~pos_ok][:5], oi[r][~pos_ok][:5])


def check_exact(table, q32, k, mask, s, i, d):
    val, oi, amb = oracle(table, q32, k, mask)
    compare_rows(lambda r, ids: val[r, ids], lambda r, ids: amb[r, ids], oi, s.cpu().numpy(), i.cpu().numpy(),
                 d.cpu().numpy())


def _setup(ccr, B, N, D, k, mode, sim, scan):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(B * 7 + N)
    P = cases.embeddings(N + 1, N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(N + 2, B, D, clustered=(sim == "cos"))
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"),
                                           dtype=SCANS[scan], exact=True)
    mask = _mask(rs, B, N, mode, dev, ccr) if mode != O.MASK_NONE else None
    return table, table.encode_queries(torch.as_tensor(Q)), mask


@pytest.mark.parametrize("scan", ["bf16", "fp16"])
@pytest.mark.parametrize("algo", [1, 2])
@pytest.mark.parametrize("B,N,D,k,mode,sim", CASES)
def test_exact_matches_float64_oracle(ccr, scan, algo, B, N, D, k, mode, sim, lever):
    table, q32, mask = _setup(ccr, B, N, D, k, mode, sim, scan)
    s, i, d, n_fb = table._search_exact(q32, k, mask=mask, algo=algo, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    check_exact(table, q32, k, mask, s, i, d)
    print(f"{scan} algo={algo} B={B} N={N} k={k}: {n_fb} fallback rows")
    # forced fallback: every row through the dense scan + compaction + re-rank, bit-identical
    lever(CCR_EXACT_FALLBACK="1")
    s2, i2, d2, n_fb2 = table._search_exact(q32, k, mask=mask, algo=algo, want_f64=True, encoded=True)
    assert n_fb2 == B
    assert torch.equal(i, i2) and torch.equal(d, d2) and torch.equal(s, s2)


@pytest.mark.parametrize("scan", ["bf16", "fp16"])
def test_certificate_fails_on_near_duplicates(ccr, scan):
    """Thousands of rows that differ below the scan format's precision but not in fp32: the scan cannot
    order them, the certificate must fail and the fallback must still give the exact ranking."""
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(5)
    D, N, n_dup, B, k = 256, 20000, 4000, 16, 100
    base = rs.standard_normal(D).astype(np.float32)
    P = rs.standard_normal((N, D)).astype(np.float32)
    P[:n_dup] = base + (rs.standard_normal((n_dup, D)) * 1e-4).astype(np.float32)
    Q = np.tile(base, (B, 1)) + (rs.standard_normal((B, D)) * 1e-3).astype(np.float32)
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, dtype=SCANS[scan], exact=True)
    q32 = table.encode_queries(torch.as_tensor(Q))
    s, i, d, n_fb = table._search_exact(q32, k, want_f64=True, encoded=True)
    assert n_fb > 0
    check_exact(table, q32, k, None, s, i, d)
    # the default (scan-format) ranking of the same table does not get these rows right
    plain = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, dtype=SCANS[scan])
    _, i_plain = plain.search(torch.as_tensor(Q), k)
    assert not torch.equal(i_plain, i)


def _adversarial(rs, kind, N, D):
    if kind == "wide_range":
        return (rs.standard_normal((N, D)) * 10.0 ** rs.uniform(-3, 3, (N, 1))).astype(np.float32)
    if kind == "cancellation":
        x = rs.standard_normal((N, D)).astype(np.float32) * 100
        x[:, D // 2 :] = -x[:, : D // 2] + rs.standard_normal((N, D // 2)).astype(np.float32) * 1e-3
        return x
    if kind == "fp16_subnormal":
        return (rs.standard_normal((N, D)) * 3e-6).astype(np.float32)
    if kind == "fp16_large":
        return (rs.standard_normal((N, D)) * 3e3).clip(-6e4, 6e4).astype(np.float32)
    raise ValueError(kind)


BOUND_SHAPES = [(B, N, D) for B, N, D, *_ in CASES] + [("wide_range", 64), ("cancellation", 64),
                                                         ("fp16_subnormal", 128), ("fp16_large", 64)]


@pytest.mark.parametrize("scan", ["bf16", "fp16"])
@pytest.mark.parametrize("shape", BOUND_SHAPES, ids=str)
def test_error_bound_holds(ccr, scan, shape):
    """Every scan score (fused kernel outputs on both algorithms, dense tiles) is within E_row of the exact
    value; prints the largest |s^ - s| / E_row."""
    from ccr_b200 import engine

    dev = torch.device("cuda:0")
    rs = np.random.RandomState(11)
    if isinstance(shape[0], str):
        kind, D = shape
        B, N = 40, 3000
        P, Q = _adversarial(rs, kind, N, D), _adversarial(rs, kind, B, D)
        Q[:, ::2] *= -1
    else:
        B, N, D = shape
        P, Q = rs.standard_normal((N, D)).astype(np.float32), rs.standard_normal((B, D)).astype(np.float32)
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, dtype=SCANS[scan], exact=True)
    q32 = table.encode_queries(torch.as_tensor(Q))
    q_scan = torch.empty(q32.shape, dtype=table.dtype, device=dev)
    table._scan_copy(q32, q_scan)
    Pd, Qd = _rows32(table, q32)
    exact = (Qd @ Pd.T).astype(np.float32).astype(np.float64)
    E = engine.exact_error_bound(np.sqrt((Qd * Qd).sum(1)), float(table.v_max.item()), table.ld, scan == "fp16")
    assert np.allclose(E, [ccr._lib.lib().ccr_exact_error_bound(float(np.sqrt((r * r).sum())), float(table.v_max.item()),
                                                                 table.ld, ccr._lib.FLAG_F16 if scan == "fp16" else 0)
                           for r in Qd], rtol=1e-12, atol=0)
    worst = 0.0
    k = min(N, 200)
    for algo in (1, 2):
        s, i = engine.score_topk(q_scan, table.data, k, algo=algo, n_items=table.n, D=table.ld)
        got = s.double().cpu().numpy()
        ref = np.take_along_axis(exact, i.cpu().numpy(), 1)
        worst = max(worst, float((np.abs(got - ref) / E[:, None]).max()))
    dense = engine.score_dense(q_scan, table.data, n_items=table.n, D=table.ld).double().cpu().numpy()
    worst = max(worst, float((np.abs(dense - exact) / E[:, None]).max()))
    print(f"{scan} {shape}: max |s^ - s| / E_row = {worst:.4f}")
    assert worst <= 1.0


def test_exact_edge_cases(ccr, tmp_path):
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(3)
    P = rs.standard_normal((50, 64)).astype(np.float32)
    Q = rs.standard_normal((3, 64)).astype(np.float32)
    for scan in SCANS.values():
        t = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, dtype=scan, exact=True)
        q32 = t.encode_queries(torch.as_tensor(Q))
        s, i, d = t.search(q32, 50, want_f64=True, encoded=True)  # k == N
        check_exact(t, q32, 50, None, s, i, d)
        with pytest.raises(RuntimeError, match="selected index k out of range"):
            t.search(torch.as_tensor(Q), 51)
        s, i = t.search(torch.zeros(0, 64), 5)
        assert s.shape == (0, 5) and i.shape == (0, 5)
        with pytest.raises(NotImplementedError):
            t.dense_scores(torch.as_tensor(Q))
        # save / load keeps the fp32 rows, V and the flag
        t.save(str(tmp_path / "t.pt"))
        u = ccr.EmbeddingTable.load(str(tmp_path / "t.pt"), device=dev)
        assert u.exact and u.dtype == scan and float(u.v_max.item()) == float(t.v_max.item())
        assert torch.equal(u.data32[: u.n], t.data32[: t.n]) and torch.equal(u.data[: u.n], t.data[: t.n])
        s2, i2 = u.search(torch.as_tensor(Q), 7)
        s1, i1 = t.search(torch.as_tensor(Q), 7)
        assert torch.equal(i1, i2) and torch.equal(s1, s2)
    # empty shard with allow_short: padded
    e = ccr.EmbeddingTable(4, 64, device=dev, exact=True)
    s, i = e.search(torch.as_tensor(Q), 5, allow_short=True)
    assert (i == -1).all() and torch.isinf(s).all()
    # all-zero table: lowest ids
    z = ccr.EmbeddingTable.from_tensor(torch.zeros(500, 64), device=dev, exact=True)
    s, i = z.search(torch.zeros(4, 64), 30)
    np.testing.assert_array_equal(i.cpu().numpy(), np.tile(np.arange(30), (4, 1)))
    # fp16 scan overflow is refused as for fp16 tables
    with pytest.raises(ValueError, match="overflow fp16"):
        ccr.EmbeddingTable.from_tensor(torch.full((3, 64), 7e4), device=dev, dtype=torch.float16, exact=True)
    # an old file (no flag) loads as a non-exact table
    plain = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev)
    plain.save(str(tmp_path / "p.pt"))
    assert not ccr.EmbeddingTable.load(str(tmp_path / "p.pt"), device=dev).exact


def _tie_aware_agreement(order, ref_order, ref_scores, tol):
    """Share of rows whose positions match the golden, counting a swap of two golden scores within tol as a
    match."""
    ok = 0
    for r in range(len(order)):
        sc = dict(zip(ref_order[r].tolist(), ref_scores[r].tolist()))
        bad = [j for j in range(order.shape[1]) if order[r, j] != ref_order[r, j]
               and not (order[r, j] in sc and abs(sc[order[r, j]] - ref_scores[r, j]) <= tol)]
        ok += not bad
    return ok / max(1, len(order))


def _profile_arrays(prof, c):
    pos = {pid: i for i, pid in enumerate(c["corpus"].keys())}
    qids = list(c["queries"].keys())
    return (np.array([[pos[p] for p in prof[q].keys()] for q in qids]),
            np.array([list(prof[q].values()) for q in qids]))


@pytest.mark.parametrize("name", list(cases.RANKING_CASES))
def test_exact_ranking_vs_cpu_golden(ccr, name, golden_dir, monkeypatch):
    """The reference's CPU ranking is fp32: with exact=True the goldens hold at 1e-5 (bf16 tables: 1e-2).

    Tolerance: rtol 1e-5 plus atol 1e-5 of the live scores' scale.  The golden is the reference's blocked fp32
    CPU matmul, not an exact sum: 768-term dot products with cancellation carry an absolute error of that
    order in small scores (DESIGN.md section 6b)."""
    import os

    g = np.load(os.path.join(golden_dir, f"ranking_{name}.npz"))
    c = cases.ranking_case(name)
    monkeypatch.setenv("CCREC_SIM_TYPE", c["sim_type"])
    run = lambda **kw: _profile_arrays(ccr.ranking(c["corpus"], c["queries"], cases.TextTable(c["table"]),  # noqa: E731
                                                   c["batch_size"], c["block_dict"], **kw), c)
    order, scores = run(table_dtype=torch.float16, exact=True)
    live = g["scores"][g["scores"] > -1e6]
    tol = 1e-5 * float(np.abs(live).max())
    errs = O.check_topk(scores, order, ref_scores=g["scores"], ref_ids=g["order"], rtol=1e-5, atol=tol)
    assert not errs, errs[:5]
    # the ordered top-2 is the golden's in every row, but for a pair of golden scores within the tolerance
    for r in range(len(order)):
        if not np.array_equal(order[r, :2], g["order"][r, :2]):
            assert abs(g["scores"][r, 0] - g["scores"][r, 1]) <= tol + 1e-5 * abs(g["scores"][r, 0]), r
    d_order, _ = run()
    print(f"{name}: tie-aware row agreement with the fp32 golden: exact "
          f"{_tie_aware_agreement(order, g['order'], g['scores'], tol):.4f}, default bf16 "
          f"{_tie_aware_agreement(d_order, g['order'], g['scores'], tol):.4f}")


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_exact_assign_topk_vs_rime_golden(ccr, name, golden_dir):
    """_assign_topk(exact=True) on the factor pair gives the reference's indices in every row, except swaps
    of two items whose scores lie within 1e-5 relative (the reference's own fp32 sums and tie jitter)."""
    import os

    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = ccr.LazyDenseMatrix(c["U"]) @ ccr.LazyDenseMatrix(c["V"]).T
    if c["prior"] is not None:
        S = S + c["prior"]
    k = c["k"]
    dense = O.lazy_score_dense_ref(c["U"], c["V"], c["prior"]).numpy().astype(np.float64)
    ref = g["indices"].reshape(len(c["U"]), k)
    agree = {}
    for exact in (True, False):
        csr = ccr._assign_topk(S, k, device="cpu", exact=exact)
        np.testing.assert_array_equal(csr.indptr, g["indptr"])
        got = csr.indices.reshape(len(c["U"]), k)
        a = np.take_along_axis(dense, got, 1)
        b = np.take_along_axis(dense, ref, 1)
        near = np.abs(a - b) <= 1e-5 * np.maximum(np.abs(a), np.abs(b)) + 1e-30
        row_ok = ((got == ref) | near).all(axis=1)
        agree[exact] = float(row_ok.mean())
        if exact:
            assert row_ok.all(), np.nonzero(~row_ok)[0][:5]
    print(f"{name}: tie-aware row agreement with the reference: exact {agree[True]:.4f}, default {agree[False]:.4f}")
    m_exact = ccr.evaluate_item_rec(sps_csr(g), S, k, exact=True)
    assert np.isfinite(m_exact["obj_mean"])


def sps_csr(g):
    import scipy.sparse as sps

    return sps.csr_matrix((g["data"], g["indices"].ravel(), g["indptr"]), shape=tuple(g["shape"]))


def _bench_workload(B, N, D, k, scan):
    """The bench workload's shape on an exact table: randn rows, a history mask of Geom(1/8) (<= 64) SET -1e6
    entries per row."""
    import ccr_b200

    g = torch.Generator(device="cuda").manual_seed(0)
    table = ccr_b200.EmbeddingTable(N, D, device="cuda", dtype=scan, exact=True)
    for s in range(0, N, 1 << 20):
        table.append(torch.randn(min(N, s + (1 << 20)) - s, D, device="cuda", generator=g))
    q32 = table.encode_queries(torch.randn(B, D, device="cuda", generator=g))
    rs = np.random.RandomState(1)
    rows = [rs.randint(0, N, size=min(64, rs.geometric(1 / 8))) for _ in range(B)]
    mask = ccr_b200.SparseMask.from_lists(rows, N, -1e6, ccr_b200.MASK_SET, "cuda")
    return table, q32, mask


def test_exact_bench_workload_fp16(ccr, lever):
    """8.84 M x 768, B = 4096, k = 100, history mask, fp16 scan: every row against an fp32 device oracle at
    1e-5, 64 rows bit-identical to a float64 device oracle, bit-identical under every lever."""
    B, N, D, k = 4096, 8841823, 768, 100
    table, q32, mask = _bench_workload(B, N, D, k, torch.float16)
    s, i, d, n_fb = table._search_exact(q32, k, mask=mask, want_f64=True, encoded=True)
    print(f"bench workload, fp16 scan: {n_fb} fallback rows")
    ip, mc, _ = mask.host
    ip_t, mc_t = torch.as_tensor(ip, device="cuda"), torch.as_tensor(mc, device="cuda").long()
    mrow = torch.repeat_interleave(torch.arange(B, device="cuda"), ip_t[1:] - ip_t[:-1])
    # fp32 device oracle (no TF32), chunked over items
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        best_v = best_i = None
        step = 1 << 20
        for c0 in range(0, N, step):
            c1 = min(N, c0 + step)
            sc = q32 @ table.data32[c0:c1].T
            sel = (mc_t >= c0) & (mc_t < c1)
            sc[mrow[sel], mc_t[sel] - c0] = -1e6
            v, ix = torch.topk(sc, k, dim=1)
            v, ix = (v, ix + c0) if best_v is None else (torch.cat([best_v, v], 1), torch.cat([best_i, ix + c0], 1))
            best_v, o = torch.topk(v, k, dim=1)
            best_i = torch.gather(ix, 1, o)
            del sc
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    errs = O.check_topk(d.cpu().numpy(), i.cpu().numpy(), ref_scores=best_v.double().cpu().numpy(),
                        ref_ids=best_i.cpu().numpy(), rtol=1e-5)
    assert not errs, errs[:5]
    # 64 rows against float64 sums, bit for bit
    rows = np.random.RandomState(2).choice(B, 64, replace=False)
    q64 = q32[torch.as_tensor(rows, device="cuda")].double()
    s64 = torch.empty((64, N), dtype=torch.float64, device="cuda")
    for c0 in range(0, N, 1 << 20):
        c1 = min(N, c0 + (1 << 20))
        s64[:, c0:c1] = q64 @ table.data32[c0:c1].double().T
    s32 = s64.float()
    val = s32.double()
    c = s32.double()
    lo = torch.nextafter(s32, torch.full_like(s32, -np.inf)).double()
    hi = torch.nextafter(s32, torch.full_like(s32, np.inf)).double()
    amb = torch.minimum((s64 - (lo + c) / 2).abs(), (s64 - (hi + c) / 2).abs()) <= s64.abs() * 2.0 ** -40
    del lo, hi, c
    for j, r in enumerate(rows):
        cols = mc_t[ip[r] : ip[r + 1]]
        val[j, cols] = -1e6
        amb[j, cols] = False
    order = torch.sort(val, dim=1, descending=True, stable=True).indices[:, :k]
    pick = (lambda t: lambda j, ids: t[j, torch.as_tensor(ids, device="cuda")].cpu().numpy())  # noqa: E731
    compare_rows(pick(val), pick(amb), order.cpu().numpy(),
                 s.cpu().numpy()[rows], i.cpu().numpy()[rows], d.cpu().numpy()[rows])
    del s64, s32, val
    for name, value in (("CCR_2CTA", "0"), ("CCR_2CTA", "1"), ("CCR_LEAD", "4"), ("CCR_NO_HIST", "1"),
                        ("CCR_EXACT_FALLBACK", "1")):
        with levers(**{name: value}):
            s2, i2, d2, _ = table._search_exact(q32, k, mask=mask, want_f64=True, encoded=True)
        assert torch.equal(i, i2) and torch.equal(d, d2) and torch.equal(s, s2), (name, value)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_exact_sharded_index_equals_one_table(world):
    """ShardedIndex(exact=True) over 2 / 4 / 8 GPUs returns what one exact table returns, bit for bit."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29900 + world + os.getpid() % 50
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(root, "tests", "dist_exact_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-4000:]
    assert r.returncode == 0, tail
    assert r.stdout.count("exact_equal_single_table=True") == 5 * world, tail
