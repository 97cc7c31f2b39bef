"""Exact dense scores (ccr_score_dense_exact, EmbeddingTable.dense_scores(exact=True), _argsort(exact=True),
cos_sim(exact=True)) bit for bit against the host emulation of dot_f64's order and against the exact re-rank's
own values.  Needs a B200."""
import os

import numpy as np
import pytest
import torch

import cases
from oracle import ccr_oracle as O
from test_exact_dense_cpu import exact_dense_values
from test_gpu_exact import _adversarial
from test_gpu_parity import CASES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


def assert_bits_equal(got, want):
    """Equal as fp32 bit patterns (+0.0 and -0.0 differ, NaN payloads count)."""
    g = got.contiguous().view(torch.int32).cpu().numpy()
    w = torch.as_tensor(want).to(got.device).contiguous().view(torch.int32).cpu().numpy()
    assert g.shape == w.shape
    bad = np.argwhere(g != w)
    assert bad.size == 0, (len(bad), bad[:5], g[tuple(bad[:5].T)], w[tuple(bad[:5].T)])


def _table(ccr, P, sim="dot"):
    return ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device="cuda", normalize=(sim == "cos"), exact=True)


def _check_table(t, q32):
    got = t.dense_scores(q32, encoded=True, exact=True)
    torch.cuda.synchronize()
    assert got.shape == (q32.shape[0], t.n)
    assert_bits_equal(got, exact_dense_values(q32, t.data32[: t.n], t.ld))
    return got


@pytest.mark.parametrize("sim", ["dot", "cos"])
@pytest.mark.parametrize("B,N,D", sorted({(B, N, D) for B, N, D, *_ in CASES}))
def test_dense_exact_equals_emulation_on_parity_shapes(ccr, B, N, D, sim):
    clustered = sim == "cos"
    t = _table(ccr, cases.embeddings(N + 1, N, D, clustered=clustered), sim)
    _check_table(t, t.encode_queries(torch.as_tensor(cases.embeddings(N + 2, B, D, clustered=clustered))))


# the kernel's block tile is 16 queries x 32 items, its K-slice 128 elements
TILE_SHAPES = [(1, 1), (15, 31), (16, 32), (17, 33), (31, 63), (32, 64), (33, 65)]


@pytest.mark.parametrize("D", [8, 64, 768, 4096])
def test_dense_exact_tile_tails(ccr, D):
    rs = np.random.RandomState(D)
    for B, N in TILE_SHAPES:
        t = _table(ccr, rs.standard_normal((N, D)).astype(np.float32))
        _check_table(t, t.encode_queries(torch.as_tensor(rs.standard_normal((B, D)).astype(np.float32))))


def test_dense_exact_pitched_inputs_ignore_columns_past_d(ccr):
    """q and items with pitches above D (NaN past D) and an output pitch above N (untouched past N)."""
    from ccr_b200 import _lib

    rs = np.random.RandomState(1)
    B, N, D, ldq, ldi, ld_out = 37, 70, 200, 224, 256, 80
    q = torch.full((B, ldq), float("nan"), device="cuda")
    items = torch.full((N, ldi), float("nan"), device="cuda")
    q[:, :D] = torch.as_tensor(rs.standard_normal((B, D)).astype(np.float32))
    items[:, :D] = torch.as_tensor(rs.standard_normal((N, D)).astype(np.float32))
    out = torch.full((B, ld_out), -7.0, device="cuda")
    rc = _lib.lib().ccr_score_dense_exact(q.data_ptr(), B, ldq, items.data_ptr(), N, ldi, D, out.data_ptr(), ld_out,
                                          torch.cuda.current_stream().cuda_stream)
    _lib.check(rc)
    torch.cuda.synchronize()
    want = exact_dense_values(q, items, D)
    assert_bits_equal(out[:, :N], want)
    assert (out[:, N:] == -7.0).all()
    from ccr_b200 import engine

    assert_bits_equal(engine.score_dense_exact(q, items, D=D), want)


@pytest.mark.parametrize("kind", ["cancellation", "wide_range", "zeros"])
def test_dense_exact_adversarial_tables(ccr, kind):
    """Cancellation, six decades of row scale, and rows of +0.0 / -0.0 (the sign of an exact zero is the
    kernel's: +0.0 for every pair)."""
    rs = np.random.RandomState(4)
    B, N, D = 40, 300, 64
    if kind == "zeros":
        P = rs.standard_normal((N, D)).astype(np.float32)
        Q = rs.standard_normal((B, D)).astype(np.float32)
        P[::3], Q[::4] = 0.0, -0.0
        P[1::7] = -0.0
        Q[1::5, : D // 2] = -0.0
    else:
        P, Q = _adversarial(rs, kind, N, D), _adversarial(rs, kind, B, D)
        Q[:, ::2] *= -1
    t = _table(ccr, P)
    got = _check_table(t, t.encode_queries(torch.as_tensor(Q)))
    if kind == "zeros":
        z = got.cpu().numpy()[::4]
        assert (z == 0).all() and not np.signbit(z).any()


def _rerank_values(t, q32, cand, k):
    """ccr_rerank_exact's float64 values [B, N] (NaN where no candidate) for candidate ids cand [B, c]."""
    from ccr_b200 import _lib

    B, c = cand.shape
    dev = q32.device
    indptr = torch.arange(B + 1, dtype=torch.int64, device=dev) * c
    ids = cand.reshape(-1).contiguous()
    out_s = torch.empty((B, k), dtype=torch.float32, device=dev)
    out_d = torch.empty((B, k), dtype=torch.float64, device=dev)
    out_i = torch.empty((B, k), dtype=torch.int64, device=dev)
    L = _lib.lib()
    ws = torch.empty(max(256, L.ccr_rerank_exact_workspace_bytes(B, B * c, 0)), dtype=torch.uint8, device=dev)
    rc = L.ccr_rerank_exact(q32.data_ptr(), B, q32.stride(0), t.data32.data_ptr(), t.n, t.ld, t.ld, k,
                            indptr.data_ptr(), ids.data_ptr(), B * c, None, None, None, 0, _lib.MASK_NONE, 0,
                            out_s.data_ptr(), out_d.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(), 0,
                            torch.cuda.current_stream().cuda_stream)
    _lib.check(rc)
    assert (out_i >= 0).all()  # every candidate came back
    vals = torch.full((B, t.n), float("nan"), dtype=torch.float64, device=dev)
    vals.scatter_(1, out_i, out_d)
    return vals


REPRO_SHAPES = sorted({(B, N, D) for B, N, D, *_ in CASES}) + [(1024, 65536, 768)]


@pytest.mark.parametrize("B,N,D", REPRO_SHAPES)
def test_dense_exact_equals_rerank_values(ccr, B, N, D):
    """The dense value of a pair is the value the exact re-rank gives it, bit for bit: every item a candidate
    where N <= CCR_MAX_K (k = N), else up to CCR_MAX_K seeded distinct candidates per row (k = their count)."""
    from ccr_b200 import _lib

    rs = np.random.RandomState(B + N)
    g = torch.Generator(device="cuda").manual_seed(B + N)
    t = ccr.EmbeddingTable(N, D, device="cuda", exact=True)
    t.append(torch.randn(N, D, device="cuda", generator=g))
    q32 = t.encode_queries(torch.randn(B, D, device="cuda", generator=g))
    dense = t.dense_scores(q32, encoded=True, exact=True)
    c = min(N, _lib.MAX_K)
    if c == N:
        cand = torch.arange(N, device="cuda").repeat(B, 1)
    else:
        cand = torch.as_tensor(np.stack([rs.choice(N, c, replace=False) for _ in range(B)]), device="cuda")
    vals = _rerank_values(t, q32, cand, c)
    got = torch.gather(dense, 1, cand)
    assert_bits_equal(got, torch.gather(vals, 1, cand).float())
    if B * N > 1 << 24:  # the large block: a few whole rows against the emulation as well
        rows = torch.as_tensor(rs.choice(B, 4, replace=False), device="cuda")
        assert_bits_equal(dense[rows], exact_dense_values(q32[rows], t.data32[: t.n], t.ld))


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_argsort_exact_vs_emulation_and_rime_golden(ccr, name, golden_dir):
    """_argsort(exact=True): the stable descending sort of the exact values plus the prior in float64, and a
    head that is the reference's but for swaps of scores within 1e-5 relative (DESIGN.md section 6b, Goldens)."""
    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = ccr.LazyDenseMatrix(c["U"]) @ ccr.LazyDenseMatrix(c["V"]).T
    if c["prior"] is not None:
        S = S + c["prior"]
    r, col = ccr._argsort(S, tie_breaker=0, exact=True)
    B, N = S.shape
    ld = -(-c["U"].shape[1] // 8) * 8
    pad = lambda a: np.pad(a, ((0, 0), (0, ld - a.shape[1])))  # noqa: E731  (the table's zero padding)
    val = exact_dense_values(pad(c["U"]), pad(c["V"]), ld).astype(np.float64)
    if c["prior"] is not None:
        val = val + c["prior"].toarray()
    order = np.argsort(-val.ravel(), kind="stable")
    np.testing.assert_array_equal(r, order // N)
    np.testing.assert_array_equal(col, order % N)
    ref = O.lazy_score_dense_ref(c["U"], c["V"], c["prior"]).numpy().astype(np.float64)
    head = len(g["argsort_rows"])
    a, b = ref[r[:head], col[:head]], ref[g["argsort_rows"], g["argsort_cols"]]
    same = (r[:head] == g["argsort_rows"]) & (col[:head] == g["argsort_cols"])
    near = np.abs(a - b) <= 1e-5 * np.maximum(np.abs(a), np.abs(b))
    assert (same | near).all(), np.nonzero(~(same | near))[0][:5]
    print(f"{name}: head positions equal to the golden: {same.mean():.4f}")


def test_cos_sim_exact(ccr):
    rs = np.random.RandomState(8)
    a = torch.as_tensor(rs.standard_normal((23, 100)).astype(np.float32))
    b = torch.as_tensor(rs.standard_normal((301, 100)).astype(np.float32) * 3)
    got = ccr.cos_sim(a, b, exact=True)
    t = ccr.EmbeddingTable.from_tensor(b, normalize=True, exact=True)
    assert_bits_equal(got, exact_dense_values(t.encode_queries(a), t.data32[: t.n], t.ld))
    # the default still scores the bf16 rounding
    assert ccr.cos_sim(a, b).shape == got.shape


def test_dense_exact_errors_and_empty_blocks(ccr):
    from ccr_b200 import engine

    rs = np.random.RandomState(9)
    P = torch.as_tensor(rs.standard_normal((50, 64)).astype(np.float32))
    Q = torch.as_tensor(rs.standard_normal((3, 64)).astype(np.float32))
    with pytest.raises(ValueError, match="exact table"):
        ccr.EmbeddingTable.from_tensor(P, device="cuda").dense_scores(Q, exact=True)
    t = ccr.EmbeddingTable.from_tensor(P, device="cuda", exact=True)
    with pytest.raises(NotImplementedError, match="exact=True"):
        t.dense_scores(Q)
    assert t.dense_scores(torch.zeros(0, 64), exact=True).shape == (0, 50)
    assert ccr.EmbeddingTable(4, 64, device="cuda", exact=True).dense_scores(Q, exact=True).shape == (3, 0)
    with pytest.raises(ValueError, match="4096"):
        engine.score_dense_exact(torch.zeros(2, 4104, device="cuda"), torch.zeros(3, 4104, device="cuda"))
    with pytest.raises(TypeError):
        engine.score_dense_exact(Q.cuda().bfloat16(), P.cuda().bfloat16())
