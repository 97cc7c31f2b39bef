"""Every launch plan of the dense and BM25 top-k entries, bit-exact against plain float64 references
(select_oracle.py, DESIGN.md section 6).  Needs a B200.

Dense (``ccr_topk_dense_f32``): the float64 matrix with the mask merged (SET: the value, ADD: double(score) +
value), ranked by the kernels' order (ord64 descending, then id ascending); NaN never ranks.  BM25
(``ccr_bm25_topk`` on synthetic indexes whose impacts are chosen freely): per query a float64 accumulator from
+0.0, each term's postings added in q_terms order, rounded to float32 and ranked the same way; every row is
checked.  Each case computes its plan from the device's SM count with the mirrors in select_oracle.py, checks it
against the size query and asserts the branch it pins; the data are laid out on the streams the plan gives."""
import numpy as np
import pytest
import torch

import select_oracle as SO
from ccr_b200 import _lib, engine
from select_oracle import lever  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

NONE, SET, ADD = SO.MASK_NONE, SO.MASK_SET, SO.MASK_ADD
FLT_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _assert_no_errors(errs, what):
    assert not errs, f"{what}: " + "; ".join(errs[:5])


# ============================================ dense ============================================

def _csr(rows):
    """[(cols, vals)] per row -> (indptr, cols int32, vals float64), columns sorted."""
    indptr, cols, vals = [0], [], []
    for c, v in rows:
        c = np.asarray(c, dtype=np.int64)
        order = np.argsort(c, kind="stable")
        assert np.unique(c).size == c.size
        cols.append(c[order])
        vals.append(np.asarray(v, dtype=np.float64)[order])
        indptr.append(indptr[-1] + c.size)
    return (np.asarray(indptr, dtype=np.int64), np.concatenate(cols).astype(np.int32),
            np.concatenate(vals).astype(np.float64))


def _random_rows(rs, B, N, max_h, mode, big_row=None):
    rows = []
    for r in range(B):
        h = big_row if r == 0 and big_row is not None else rs.randint(0, max_h + 1)
        c = rs.choice(N, size=min(h, N), replace=False)
        v = rs.standard_normal(c.size) * 3 if mode == ADD else rs.choice([-1e6, 1e6, 0.5, -2.0], size=c.size)
        rows.append((c, v))
    return rows


def _dense_oracle(scores, k, csr, mode):
    full = scores.double().clone()
    if csr is not None:
        ip, cols, vals = csr
        B = scores.shape[0]
        r = torch.as_tensor(np.repeat(np.arange(B), np.diff(ip)), device=scores.device)
        c = torch.as_tensor(cols.astype(np.int64), device=scores.device)
        v = torch.as_tensor(vals, device=scores.device)
        full[r, c] = v if mode == SET else full[r, c] + v
    want_v, want_i = SO.exact_topk(full, k, drop_nan=True)
    return want_v.cpu().numpy(), want_i.cpu().numpy()


def _run_dense(scores, k, csr=None, mode=NONE, h=None):
    """engine.topk_dense on ``scores`` (a possibly strided fp32 view) with the CSR mask and row bound h (None:
    the CSR's own maximum); asserts that the size query is the mirror's total.  Returns (plan, s, i, d)."""
    B, N = scores.shape
    mask, nnz, hh = None, 0, 0
    if csr is not None and int(csr[0][-1]) > 0:
        ip, cols, vals = csr
        hh = int(np.diff(ip).max()) if h is None else h
        d = scores.device
        mask = engine.SparseMask.from_device_tensors(
            torch.as_tensor(ip, device=d), torch.as_tensor(cols, device=d), torch.as_tensor(vals, device=d),
            (ip, cols, vals), N, mode, max_row_nnz=hh)
        nnz = int(ip[-1])
    plan = SO.dense_plan(B, N, k, nnz, hh, sms=_sms())
    assert _lib.lib().ccr_topk_dense_workspace_bytes(B, N, k, nnz, hh) == plan["total"]
    s, i, d = engine.topk_dense(scores, k, mask=mask)
    torch.cuda.synchronize()
    return plan, s.cpu().numpy(), i.cpu().numpy(), d.cpu().numpy()


def _check_dense(scores, k, csr=None, mode=NONE, h=None):
    plan, s, i, d = _run_dense(scores, k, csr, mode, h)
    want_v, want_i = _dense_oracle(scores, k, csr, mode)
    _assert_no_errors(SO.check_exact(s, i, d, want_v, want_i), "dense top-k")
    return plan


def _row_nnz(csr, B):
    return np.zeros(B, np.int64) if csr is None else np.diff(csr[0])


def _case_split_cap(rs, dev):
    B, N, k = 1, 4_300_000, 2048
    x = torch.as_tensor(rs.standard_normal((B, N)).astype(np.float32), device=dev)
    plan = _check_dense(x, k)
    cols = SO.dense_split_cols(plan, N)
    assert plan["S"] == 1024, plan                      # finalize's stream cap
    assert cols[-1][0] == cols[-1][1] == N              # empty trailing splits
    assert SO.dense_finalize_entries(plan, N, k)[0] > SO.FIN_LIST   # the select runs over global memory


def _case_exclude_top(rs, dev):
    """Each row's top k + 64 values lie in one split; 48 of the row's own top columns are masked away (ADD -inf /
    -1e10) and 16 low columns boosted by +1e5, so the answer holds the row's ranks 49 .. k + 32.  The split must
    keep k + nnz(row) candidates: its 4096 values are 1 + m / 4096, 16 per histogram bucket, so a prune asked for
    only k keeps at most k + 15 and loses the answer's last ranks."""
    B, N, k, h = 7, 300_000, 1001, 64
    plan = SO.dense_plan(B, N, k, B * h, h, sms=_sms())
    full = [s for s, (a, b) in enumerate(SO.dense_split_cols(plan, N)) if b - a == SO.DENSE_SLACK]
    x = rs.uniform(-1.0, 0.99, size=(B, N)).astype(np.float32)
    rows = []
    for r in range(B):
        a = SO.dense_split_cols(plan, N)[full[(3 * r + 1) % len(full)]][0]
        x[r, a : a + SO.DENSE_SLACK] = 1.0 + rs.permutation(SO.DENSE_SLACK) / SO.DENSE_SLACK
        top = np.argsort(-x[r], kind="stable")[:48]
        assert np.all((top >= a) & (top < a + SO.DENSE_SLACK))
        low = rs.choice(np.nonzero(x[r] < 0)[0], size=16, replace=False)
        rows.append((np.concatenate([top, low]),
                     np.concatenate([np.tile([-np.inf, -1e10], 24), 1e5 + rs.standard_normal(16)])))
    csr = _csr(rows)
    plan = _check_dense(torch.as_tensor(x, device=dev), k, csr, ADD)
    assert 1 < plan["S"] < SO.FIN_MAX_STREAMS and plan["per"] == SO.DENSE_SLACK
    assert plan["C"] - SO.DENSE_SLACK < SO.DENSE_SLACK   # the split prunes after its one chunk
    assert SO.dense_finalize_entries(plan, N, k + h, h)[0] > SO.FIN_LIST


def _case_kh_2048(rs, dev):
    B, N, k = 2000, 4096, 2000
    csr = _csr(_random_rows(rs, B, N, 48, SET, big_row=48))
    x = torch.as_tensor(rs.standard_normal((B, N)).astype(np.float32), device=dev)
    plan = _check_dense(x, k, csr, SET)
    assert plan["S"] == 1 and plan["k_keep"] == _lib.MAX_K
    for nnz in set(_row_nnz(csr, B).tolist()):   # no prune: exactly the shared list's capacity reaches finalize
        assert SO.dense_finalize_entries(plan, N, k + nnz, nnz) == (SO.FIN_LIST, SO.FIN_LIST)


def _case_bound_h(rs, dev):
    """SET on each row's top 20 columns (half -1e6, half above every score) with max_row_nnz = 300: buffers
    sized by the bound; finalize in shared memory must drop those columns' stream candidates."""
    B, N, k = 40, 20_000, 100
    x = rs.standard_normal((B, N)).astype(np.float32)
    rows = []
    for r in range(B):
        top = np.argsort(-x[r], kind="stable")[:20]
        rows.append((top, np.where(np.arange(20) % 2 == 0, -1e6, 10.0 + rs.standard_normal(20))))
    csr = _csr(rows)
    plan = _check_dense(torch.as_tensor(x, device=dev), k, csr, SET, h=300)
    assert plan["k_keep"] == k + 300 and plan["S"] > 1
    assert SO.dense_finalize_entries(plan, N, k + 20, 20)[1] <= SO.FIN_LIST


def _case_unaligned(rs, dev):
    B, N, k = 300, 20_011, 10
    buf = torch.empty(1 + B * (N + 1), dtype=torch.float32, device=dev)
    x = buf[1:].view(B, N + 1)[:, :N]
    x.copy_(torch.as_tensor(rs.standard_normal((B, N)).astype(np.float32)))
    x[::3] = torch.as_tensor(rs.randint(0, 50, size=x[::3].shape).astype(np.float32), device=dev)
    assert x.stride(0) == N + 1 and x.data_ptr() % 16 == 4
    plan = _check_dense(x, k, _csr(_random_rows(rs, B, N, 30, ADD)), ADD)
    assert N % SO.DENSE_SLACK != 0 and plan["S"] > 1


def _case_k_eq_n(rs, dev):
    B, N, k = 5, 37, 37
    rows = [(c, np.full(c.size, -1e30)) for c, _ in _random_rows(rs, B, N, 10, SET)]
    _check_dense(torch.as_tensor(rs.standard_normal((B, N)).astype(np.float32), device=dev), k, _csr(rows), SET)


def _case_k_plus_h_over_n(rs, dev):
    B, N, k, h = 3, 50, 40, 30
    rows = [(rs.choice(N, size=h, replace=False), np.full(h, -1e30)) for _ in range(B)]
    x = torch.as_tensor(rs.standard_normal((B, N)).astype(np.float32), device=dev)
    plan = _check_dense(x, k, _csr(rows), SET)
    assert plan["k_keep"] > N


def _old_shape(B, N, k, mode):
    """The shapes of the former float64-sort test: every third row drawn from 50 integer values."""
    def case(rs, dev):
        x = rs.standard_normal((B, N)).astype(np.float32)
        x[::3] = rs.randint(0, 50, size=x[::3].shape).astype(np.float32)
        csr = _csr(_random_rows(rs, B, N, min(N, 30), mode)) if mode != NONE else None
        _check_dense(torch.as_tensor(x, device=dev), k, csr, mode)
    return case


DENSE_CASES = {
    "d-split-cap": _case_split_cap,
    "d-exclude-top": _case_exclude_top,
    "d-kh-2048": _case_kh_2048,
    "d-bound-h": _case_bound_h,
    "d-unaligned": _case_unaligned,
    "d-kN": _case_k_eq_n,
    "d-k+h>N": _case_k_plus_h_over_n,
    "d-7x5000-k100": _old_shape(7, 5000, 100, NONE),
    "d-300x20000-k1001-add": _old_shape(300, 20_000, 1001, ADD),
    "d-2x300000-k10-set": _old_shape(2, 300_000, 10, SET),
    "d-40x37-k37-add": _old_shape(40, 37, 37, ADD),
    "d-1100x3000-k5": _old_shape(1100, 3000, 5, NONE),
}


@pytest.mark.parametrize("case", list(DENSE_CASES))
def test_dense_plan_case(case, dev):
    DENSE_CASES[case](np.random.RandomState(sum(map(ord, case))), dev)


def test_dense_k_out_of_range(dev):
    with pytest.raises(RuntimeError, match="out of range"):
        engine.topk_dense(torch.zeros(2, 3, device=dev), 4)


LAYOUTS = ["normal", "ascending", "descending", "top-in-last-split", "all-equal", "tie-run", "mostly-inf",
           "specials", "negative", "integers"]


def _layout_row(name, rs, N, k, last):
    if name == "normal":
        return rs.standard_normal(N)
    if name == "ascending":
        return np.arange(N) / N
    if name == "descending":
        return 1.0 - np.arange(N) / N
    if name == "top-in-last-split":
        x = rs.standard_normal(N) - 10
        x[rs.choice(np.arange(*last), size=3 * k // 2, replace=False)] += 20
        return x
    if name == "all-equal":
        return np.full(N, 0.5)
    if name == "tie-run":   # k-th rank inside a run of ~N ties
        x = np.ones(N)
        x[rs.choice(N, size=k // 2, replace=False)] = 2.0
        return x
    if name == "mostly-inf":   # fewer than k finite values: -inf entries at the lowest columns complete the answer
        x = np.full(N, -np.inf)
        x[rs.choice(N, size=k * 3 // 5, replace=False)] = rs.standard_normal(k * 3 // 5)
        return x
    if name == "specials":
        sub = float(np.finfo(np.float32).smallest_subnormal)
        return rs.choice([np.inf, -np.inf, FLT_MAX, -FLT_MAX, sub, -sub, 4 * sub, 0.0, -0.0, 1.0], size=N)
    if name == "negative":
        return -np.abs(rs.standard_normal(N)) - 1e-3
    if name == "integers":
        return rs.randint(0, 50, size=N)
    raise KeyError(name)


@pytest.mark.parametrize("B", [64, 1184])
@pytest.mark.parametrize("mode", [NONE, ADD])
def test_dense_score_layouts(mode, B, dev):
    """N = 40,000, k = 100; row r has layout r % 10 (streaming thresholds: most prunes, failed block votes, late
    winners, the exact-select fallback on ties, -inf keys below the histogram clamp, specials).  B = 64: ten
    one-chunk splits on 148 SMs; B = 1184: one split of ten chunks, whose threshold each chunk must pass."""
    N, k = 40_000, 100
    rs = np.random.RandomState(11 + mode + B)
    plan = SO.dense_plan(B, N, k, sms=_sms())
    last = [c for c in SO.dense_split_cols(plan, N) if c[1] > c[0]][-1]
    x = np.stack([_layout_row(LAYOUTS[r % len(LAYOUTS)], rs, N, k, last) for r in range(B)]).astype(np.float32)
    csr = _csr(_random_rows(rs, B, N, 30, ADD)) if mode == ADD else None
    plan = _check_dense(torch.as_tensor(x, device=dev), k, csr, mode)
    assert plan["S"] > 1 if B == 64 else plan["per"] > SO.DENSE_SLACK


@pytest.mark.parametrize("mode", [NONE, SET, ADD])
def test_dense_nan_never_ranks(mode, dev):
    """NaN scores (either sign) are never returned; a row with fewer than k other values ends in (-inf, -1)
    padding; an ADD mask entry on a NaN cell is NaN and never ranks either, a SET entry there ranks by its value."""
    B, N, k = 16, 10_000, 100
    rs = np.random.RandomState(5 + mode)
    x = rs.standard_normal((B, N)).astype(np.float32)
    neg_nan = np.copysign(np.float32(np.nan), np.float32(-1.0))
    for r in range(B):
        if r % 2:
            x[r, rs.choice(N, size=N // 10, replace=False)] = np.nan
            x[r, rs.choice(N, size=N // 10, replace=False)] = neg_nan
        else:   # fewer than k non-NaN values
            keep = rs.choice(N, size=k // 2, replace=False)
            y = np.full(N, np.nan, dtype=np.float32)
            y[keep] = x[r, keep]
            x[r] = y
    csr = None
    if mode != NONE:
        rows = []
        for r in range(B):
            nan_cols = np.nonzero(np.isnan(x[r]))[0]
            c = np.concatenate([rs.choice(nan_cols, size=8, replace=False),
                                rs.choice(np.nonzero(~np.isnan(x[r]))[0], size=4, replace=False)])
            rows.append((c, rs.standard_normal(12) * 3 + (5.0 if mode == ADD else 0.0)))
        csr = _csr(rows)
    _check_dense(torch.as_tensor(x, device=dev), k, csr, mode)


# ============================================ BM25 ============================================

class Index:
    """A synthetic posting index on the device: per term a doc-sorted list and freely chosen float64 impacts."""

    def __init__(self, N, terms, dev, head=()):
        self.N = N
        lens = [len(d) for d, _ in terms]
        self.indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        self.docs = np.concatenate([np.asarray(d, np.int64) for d, _ in terms] + [np.zeros(0, np.int64)])
        self.vals = np.concatenate([np.asarray(v, np.float64) for _, v in terms] + [np.zeros(0)])
        for d, _ in terms:
            assert np.all(np.diff(d) > 0) and (len(d) == 0 or (d[0] >= 0 and d[-1] < N))
        self.d_indptr = torch.as_tensor(self.indptr, device=dev)
        self.d_docs = torch.as_tensor(self.docs.astype(np.int32) if self.docs.size else np.zeros(1, np.int32), device=dev)
        self.d_vals = torch.as_tensor(self.vals if self.vals.size else np.zeros(1), device=dev)
        self.head = None
        if len(head):
            L = _lib.lib()
            n_terms = len(terms)
            slot = torch.empty(n_terms, dtype=torch.int32, device=dev)
            rows = torch.empty((len(head), int(L.ccr_bm25_head_row_pitch(N))), dtype=torch.float64, device=dev)
            d_head = torch.as_tensor(np.asarray(head, np.int32), device=dev)
            _lib.check(L.ccr_bm25_build_head_rows(self.d_indptr.data_ptr(), self.d_docs.data_ptr(),
                                                  self.d_vals.data_ptr(), d_head.data_ptr(), len(head), n_terms, N,
                                                  slot.data_ptr(), rows.data_ptr(), None))
            torch.cuda.synchronize()
            self.head = (slot, rows)


def _queries(qs):
    """[[term, ...]] -> (q_indptr, q_terms, longest)."""
    ip = np.concatenate([[0], np.cumsum([len(q) for q in qs])]).astype(np.int64)
    t = np.concatenate([np.asarray(q, np.int64) for q in qs] + [np.zeros(0, np.int64)]).astype(np.int32)
    return ip, t, max((len(q) for q in qs), default=0)


def _run_bm25(index, qs, k, use_head=True):
    L = _lib.lib()
    dev = index.d_indptr.device
    ip, t, longest = _queries(qs)
    Bq, N = len(qs), index.N
    d_ip = torch.as_tensor(ip, device=dev)
    d_t = torch.as_tensor(t if t.size else np.zeros(1, np.int32), device=dev)
    need = L.ccr_bm25_topk_workspace_bytes(Bq, N, k)
    assert need == SO.bm25_workspace(Bq, N, k, sms=_sms())
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    s = torch.empty((Bq, k), dtype=torch.float32, device=dev)
    i = torch.empty((Bq, k), dtype=torch.int64, device=dev)
    hs, hr = (index.head[0].data_ptr(), index.head[1].data_ptr()) if use_head and index.head else (None, None)
    _lib.check(L.ccr_bm25_topk(index.d_indptr.data_ptr(), index.d_docs.data_ptr(), index.d_vals.data_ptr(), hs, hr,
                               d_ip.data_ptr(), d_t.data_ptr(), longest, Bq, N, k, s.data_ptr(), i.data_ptr(),
                               ws.data_ptr(), need, None))
    torch.cuda.synchronize()
    del ws
    return s.cpu().numpy(), i.cpu().numpy()


def _bm25_f32(index, qs):
    ip, t, _ = _queries(qs)
    return SO.bm25_scores(index.indptr, index.docs, index.vals, ip, t, index.N, device=index.d_indptr.device).float()


def _check_bm25(index, qs, k, got, scores32=None):
    s, i = got
    f32 = _bm25_f32(index, qs) if scores32 is None else scores32
    want_v, want_i = SO.exact_topk(f32, k)
    _assert_no_errors(SO.check_exact(s, i, s.astype(np.float64), want_v.cpu().numpy(), want_i.cpu().numpy()),
                      "bm25 top-k")


def _run_both_kernels(lever, index, qs, k, check=True, scores32=None):  # noqa: F811
    """The warp-private kernel (auto) and the block-wide one (lever): bit-identical, and equal to the oracle."""
    lever(CCR_BM25_BLOCKWIDE=None)
    a = _run_bm25(index, qs, k)
    lever(CCR_BM25_BLOCKWIDE="1")
    b = _run_bm25(index, qs, k)
    lever(CCR_BM25_BLOCKWIDE=None)
    assert np.array_equal(a[0].view(np.int32), b[0].view(np.int32)) and np.array_equal(a[1], b[1])
    if check:
        _check_bm25(index, qs, k, a, scores32)
    return a


def _ord32(t):
    b = t.contiguous().view(torch.int32).to(torch.int64)
    return torch.where(b < 0, (~b) & 0xFFFFFFFF, b | 0x80000000)


def _sketch_row_bound(f32_row, plan, k):
    """ord32 row bound of the warp-private kernel when no stream prunes: per block the 5th largest of its 8
    streams' ceil(k/5)-th best scores (0 for a stream with fewer docs), the maximum over the blocks."""
    j = -(-k // SO.BMW_SKETCH_M)
    o = _ord32(f32_row)
    jth = []
    for a, b in SO.bm25_stream_docs(plan, f32_row.numel()):
        jth.append(int(torch.topk(o[a:b], j).values[-1]) if b - a >= j else 0)
    best = 0
    for blk in range(plan["S"]):
        v = sorted((x for x in jth[blk * SO.BMW_WARPS:(blk + 1) * SO.BMW_WARPS] if x), reverse=True)
        if len(v) >= SO.BMW_SKETCH_M:
            best = max(best, v[SO.BMW_SKETCH_M - 1])
    return best


def _random_terms(rs, N, n_terms, df_lo, df_hi, lo=0.1, hi=3.0):
    out = []
    for _ in range(n_terms):
        df = rs.randint(df_lo, df_hi + 1)
        d = np.sort(rs.choice(N, size=min(df, N), replace=False))
        out.append((d, rs.uniform(lo, hi, size=d.size)))
    return out


def test_bm25_cap_1024_streams(dev, lever):  # noqa: F811
    """One query over 10^6 docs, k = 2048: 128 blocks x 8 warps = finalize's 1024-stream cap; no stream prunes,
    the row bound is the end-of-kernel sketch and more than 4096 entries reach finalize (global memory)."""
    N, k = 1_000_000, 2048
    rs = np.random.RandomState(1)
    index = Index(N, _random_terms(rs, N, 4, 100_000, 300_000), dev)
    qs = [[0, 1, 2, 3]]
    plan = SO.bm25_plan(1, N, k, True, sms=_sms())
    assert plan["streams"] == SO.FIN_MAX_STREAMS and plan["per"] <= plan["C"] - SO.BMW_MINI
    f32 = _bm25_f32(index, qs)
    _run_both_kernels(lever, index, qs, k, scores32=f32)
    tau = _sketch_row_bound(f32[0], plan, k)
    assert int((_ord32(f32[0]) >= tau).sum()) > SO.FIN_LIST


def _concentrated(rs, N, plan, n_q, k, top_streams_of):
    """One term per query: its top k docs split evenly over 4 streams of one block, the block's other 4 streams
    holding 400 docs of lower scores each, plus 20,000 low background docs anywhere else."""
    docs_of = SO.bm25_stream_docs(plan, N)
    terms = []
    for q in range(n_q):
        streams = top_streams_of(q)
        top = np.concatenate([rs.choice(np.arange(*docs_of[s]), size=k // 4 + (i < k % 4), replace=False)
                              for i, s in enumerate(streams[:4])])
        mid = np.concatenate([rs.choice(np.arange(*docs_of[s]), size=400, replace=False) for s in streams[4:]])
        used = np.zeros(N, bool)
        used[top] = used[mid] = True
        bg = rs.choice(np.nonzero(~used)[0], size=20_000, replace=False)
        d = np.concatenate([top, mid, bg])
        v = np.concatenate([100 + rs.uniform(0, 1, top.size), 50 + rs.uniform(0, 1, mid.size),
                            rs.uniform(0, 10, bg.size)])
        order = np.argsort(d)
        terms.append((d[order], v[order]))
    return terms


def test_bm25_sketch_one_mini_chunk_per_stream(dev, lever):  # noqa: F811
    """Streams of one mini-chunk never prune: the row bound is the end-of-kernel sketch alone, and only the 5th
    largest of the 8 streams' ceil(k/5)-th best is sound when the query's top k sit in 4 streams of a block."""
    Bq, N, k = 4, 300_000, 1001
    rs = np.random.RandomState(2)
    plan = SO.bm25_plan(Bq, N, k, True, sms=_sms())
    assert plan["per"] == SO.BMW_MINI and plan["per"] <= plan["C"] - SO.BMW_MINI and plan["S"] > 4
    blocks = [b for b in range(plan["S"]) if (b + 1) * SO.BMW_WARPS * SO.BMW_MINI <= N]
    terms = _concentrated(rs, N, plan, Bq, k, lambda q: [blocks[(5 + 17 * q) % len(blocks)] * 8 + w
                                                         for w in (0, 2, 4, 6, 1, 3, 5, 7)])
    _run_both_kernels(lever, Index(N, terms, dev), [[q] for q in range(Bq)], k)


def test_bm25_sketch_in_loop(dev, lever):  # noqa: F811
    """One block per query: 8 long streams that prune many times, sharing s_tau_blk and the in-loop sketch; the
    query's top k are spread over 4 of them."""
    Bq, N, k = 600, 300_000, 1001
    rs = np.random.RandomState(3)
    plan = SO.bm25_plan(Bq, N, k, True, sms=_sms())
    assert plan["S"] == 1 and plan["per"] > 8 * plan["C"]
    terms = _concentrated(rs, N, plan, Bq, k, lambda q: list(np.roll([0, 2, 4, 6], q % 4)) + [1, 3, 5, 7])
    _run_both_kernels(lever, Index(N, terms, dev), [[q] for q in range(Bq)], k)


def test_bm25_float32_ties(dev, lever):  # noqa: F811
    """Single-term queries whose postings all carry one value (df >> k), and pairs of terms whose sums are
    distinct in float64 but equal in float32: the k-th rank lies in a run of thousands of ties, the row bound
    equals the tied value."""
    Bq, N, k = 300, 200_000, 100
    rs = np.random.RandomState(4)
    assert SO.bm25_plan(Bq, N, k, True, sms=_sms())["streams"] > 1
    terms, qs = [], []
    for q in range(Bq):
        d = np.sort(rs.choice(N, size=5000, replace=False))
        if q % 2 == 0:
            terms.append((d, np.full(d.size, 1.25)))
            qs.append([len(terms) - 1])
        else:
            sub = np.sort(rs.choice(d, size=3000, replace=False))
            terms += [(d, np.full(d.size, 1.0)), (sub, rs.uniform(1e-9, 2e-9, sub.size))]
            qs.append([len(terms) - 2, len(terms) - 1])
    _run_both_kernels(lever, Index(N, terms, dev), qs, k)


def test_bm25_head_rows(dev, lever):  # noqa: F811
    """Stop-word terms (df >= 25 %) as dense head rows, N not a multiple of 512: both kernels, with and without
    the head rows, bit-identical to the oracle; a batch with a 40-term query takes the block-wide kernel."""
    Bq, N, k = 64, 33_333, 1001
    rs = np.random.RandomState(5)
    terms = _random_terms(rs, N, 5, N // 4, 3 * N // 5) + _random_terms(rs, N, 295, 50, 3000)
    index = Index(N, terms, dev, head=list(range(5)))
    qs = [sorted(set(rs.choice(5, size=rs.randint(0, 4)).tolist()) |
                 set(rs.choice(np.arange(5, 300), size=rs.randint(1, 29)).tolist())) for _ in range(Bq)]
    assert max(map(len, qs)) <= SO.BMW_MAX_TERMS
    got = _run_both_kernels(lever, index, qs, k)
    plain = _run_bm25(index, qs, k, use_head=False)
    assert np.array_equal(got[0].view(np.int32), plain[0].view(np.int32)) and np.array_equal(got[1], plain[1])
    long_qs = qs[:8] + [list(range(0, 40))]
    a, b = _run_bm25(index, long_qs, k), _run_bm25(index, long_qs, k, use_head=False)
    assert np.array_equal(a[0].view(np.int32), b[0].view(np.int32)) and np.array_equal(a[1], b[1])
    _check_bm25(index, long_qs, k, a)


def test_bm25_blockwide_long_queries(dev):
    """Queries of 33 and 512 distinct terms over 2.1 M docs: the block-wide kernel with one split per 4096-doc
    chunk group (370 splits on 148 SMs)."""
    Bq, N, k = 2, 2_100_000, 1001
    rs = np.random.RandomState(6)
    index = Index(N, _random_terms(rs, N, 512, 500, 20_000), dev)
    qs = [sorted(rs.choice(512, size=33, replace=False).tolist()), list(range(512))]
    plan = SO.bm25_plan(Bq, N, k, False, sms=_sms())
    assert plan["S"] == min(-(-5 * _sms() // Bq), -(-N // SO.BM_CHUNK), SO.FIN_MAX_STREAMS) and plan["S"] > 1
    _check_bm25(index, qs, k, _run_bm25(index, qs, k))


@pytest.mark.parametrize("Bq,N,k", [(65535, 600, 10), (5, 511, 511), (5, 1, 1)])
def test_bm25_edges(Bq, N, k, dev, lever):  # noqa: F811
    """The largest batch (its workspace is about 2.4 GB), k = N, N below one mini-chunk; queries with no terms or
    only empty posting lists return positions 0 .. k-1 at +0.0."""
    rs = np.random.RandomState(Bq + N)
    terms = _random_terms(rs, N, 40, 1, max(1, N // 3)) + [(np.zeros(0, np.int64), np.zeros(0))] * 3
    qs = [sorted(rs.choice(40, size=rs.randint(1, 6), replace=False).tolist()) for _ in range(Bq)]
    qs[0], qs[1] = [], [40, 41, 42]
    plan = SO.bm25_plan(Bq, N, k, True, sms=_sms())
    assert plan["streams"] == SO.BMW_WARPS
    s, i = _run_both_kernels(lever, Index(N, terms, dev), qs, k)
    assert np.array_equal(i[:2], np.tile(np.arange(k), (2, 1)))
    assert np.array_equal(s[:2].view(np.int32), np.zeros((2, k), np.int32))
