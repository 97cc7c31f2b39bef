"""One rule for the sparse mask in every C entry point that takes one: a mask applies exactly when its mode is
set, indptr is given and nnz > 0.  Needs a B200.

Every data pointer handed to the library is a real device buffer of the right size, also in the calls that
must be rejected: a call that is wrongly accepted then reads valid memory."""
import numpy as np
import pytest
import torch

from select_oracle import lever  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

B, N, D, K = 4, 1024, 64, 8
ENTRY_POINTS = ["ccr_score_topk_bf16", "ccr_topk_dense_f32", "ccr_argsort_scores_f32", "ccr_score_topk_exact",
                "ccr_rerank_exact"]


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


@pytest.fixture(scope="module")
def abi(ccr):
    """(entry point name -> run(indptr, cols, vals, nnz, mode) -> (rc, outputs), the mask's device arrays).
    Every argument but the mask is fixed; the mask has 3 entries, at most 2 in one row."""
    from ccr_b200 import _lib

    L = _lib.lib()
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(7)
    q = torch.randn(B, D, generator=g).to(dev).bfloat16()
    items = torch.randn(N, D, generator=g).to(dev).bfloat16()
    q32, items32 = q.float(), items.float()
    scores = torch.randn(B, N, generator=g).to(dev)
    v_max = items32.double().norm(dim=1).max().reshape(1) * (1 + 2.0 ** -20)
    mask = (torch.tensor([0, 1, 1, 3, 3], dtype=torch.int64, device=dev),
            torch.tensor([5, 2, 700], dtype=torch.int32, device=dev),
            torch.tensor([-1e6, -1e6, -1e6], dtype=torch.float64, device=dev))
    nnz, h_max = 3, 2
    cand_indptr = torch.arange(0, 2 * B + 1, 2, dtype=torch.int64, device=dev)
    cand_ids = torch.tensor([1, 5, 2, 3, 8, 700, 9, 10], dtype=torch.int64, device=dev)
    ws_bytes = max(L.ccr_score_topk_workspace_bytes(B, N, D, K, nnz, h_max, 0),
                   L.ccr_topk_dense_workspace_bytes(B, N, K, nnz, h_max),
                   L.ccr_argsort_workspace_bytes(B * N),
                   L.ccr_score_topk_exact_workspace_bytes(B, N, D, K, nnz, h_max, 0),
                   L.ccr_rerank_exact_workspace_bytes(B, cand_ids.numel(), nnz))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream

    def outputs(*shapes_dtypes):
        return [torch.zeros(s, dtype=t, device=dev) for s, t in shapes_dtypes]

    topk = ((B, K), torch.float32), ((B, K), torch.float64), ((B, K), torch.int64)

    def score_topk_bf16(ip, c, v, n, mode):
        o = outputs(*topk)
        return L.ccr_score_topk_bf16(q.data_ptr(), B, D, items.data_ptr(), N, D, D, K, ip, c, v, n, h_max, mode, 0,
                                     o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), ws.data_ptr(), ws_bytes, 0,
                                     st), o

    def topk_dense(ip, c, v, n, mode):
        o = outputs(*topk)
        return L.ccr_topk_dense_f32(scores.data_ptr(), B, N, N, K, ip, c, v, n, h_max, mode, o[0].data_ptr(),
                                    o[1].data_ptr(), o[2].data_ptr(), ws.data_ptr(), ws_bytes, st), o

    def argsort(ip, c, v, n, mode):
        o = outputs(((B * N,), torch.int64), ((B * N,), torch.int64))
        return L.ccr_argsort_scores_f32(scores.data_ptr(), B, N, N, ip, c, v, n, mode, o[0].data_ptr(),
                                        o[1].data_ptr(), ws.data_ptr(), ws_bytes, st), o

    def score_topk_exact(ip, c, v, n, mode):
        o = outputs(*topk, ((B,), torch.int32), ((B,), torch.float64), ((1,), torch.int32))
        return L.ccr_score_topk_exact(q32.data_ptr(), q.data_ptr(), B, D, items32.data_ptr(), items.data_ptr(), N, D,
                                      D, K, v_max.data_ptr(), ip, c, v, n, h_max, mode, 0, o[0].data_ptr(),
                                      o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), o[4].data_ptr(),
                                      o[5].data_ptr(), ws.data_ptr(), ws_bytes, 0, st), o

    def rerank_exact(ip, c, v, n, mode):
        o = outputs(*topk)
        return L.ccr_rerank_exact(q32.data_ptr(), B, D, items32.data_ptr(), N, D, D, K, cand_indptr.data_ptr(),
                                  cand_ids.data_ptr(), cand_ids.numel(), ip, c, v, n, mode, 0, o[0].data_ptr(),
                                  o[1].data_ptr(), o[2].data_ptr(), ws.data_ptr(), ws_bytes, 0, st), o

    runs = dict(zip(ENTRY_POINTS, (score_topk_bf16, topk_dense, argsort, score_topk_exact, rerank_exact)))
    return runs, mask


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_every_entry_point_rejects_the_same_bad_masks(ccr, abi, name):
    from ccr_b200 import _lib

    runs, (ip, c, v) = abi
    run = runs[name]
    assert run(ip.data_ptr(), c.data_ptr(), v.data_ptr(), 3, 7)[0] == _lib.EINVAL
    assert run(ip.data_ptr(), None, v.data_ptr(), 3, ccr.MASK_SET)[0] == _lib.EINVAL
    assert run(ip.data_ptr(), c.data_ptr(), v.data_ptr(), -1, ccr.MASK_SET)[0] == _lib.EINVAL
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_empty_mask_without_cols_and_vals_is_no_mask(ccr, abi, name):
    from ccr_b200 import _lib

    runs, (ip, _, _) = abi
    empty_ip = torch.zeros_like(ip)
    rc, got = runs[name](empty_ip.data_ptr(), None, None, 0, ccr.MASK_SET)
    rc_ref, ref = runs[name](None, None, None, 0, ccr.MASK_NONE)
    torch.cuda.synchronize()
    assert rc == rc_ref == _lib.OK
    for a, b in zip(got, ref):
        assert torch.equal(a, b)


def _empty_set_mask(ccr, n_rows, n_cols):
    return ccr.SparseMask.from_lists([[]] * n_rows, n_cols, -1e6, ccr.MASK_SET, torch.device("cuda:0"))


def _same(a, b):
    assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("algo", [1, 2])
def test_score_topk_empty_mask_equals_no_mask(ccr, algo, dtype):
    rs = np.random.RandomState(11)
    P = torch.as_tensor(rs.standard_normal((3000, 128)).astype(np.float32))
    Q = torch.as_tensor(rs.standard_normal((5, 128)).astype(np.float32))
    table = ccr.EmbeddingTable.from_tensor(P, device=torch.device("cuda:0"), dtype=dtype)
    empty = _empty_set_mask(ccr, 5, 3000)
    _same(table.search(Q, 50, mask=empty, algo=algo, want_f64=True), table.search(Q, 50, algo=algo, want_f64=True))


def test_dense_wrappers_empty_mask_equals_no_mask(ccr):
    from ccr_b200 import engine

    scores = torch.randn(6, 2000, generator=torch.Generator().manual_seed(3)).cuda()
    empty = _empty_set_mask(ccr, 6, 2000)
    _same(engine.topk_dense(scores, 40, mask=empty), engine.topk_dense(scores, 40))
    _same(engine.argsort_scores(scores, mask=empty), engine.argsort_scores(scores))


@pytest.mark.parametrize("fallback", [False, True])
def test_score_topk_exact_empty_mask_equals_no_mask(ccr, lever, fallback):
    if fallback:
        lever(CCR_EXACT_FALLBACK="1")
    rs = np.random.RandomState(13)
    P = torch.as_tensor(rs.standard_normal((3000, 128)).astype(np.float32))
    Q = torch.as_tensor(rs.standard_normal((5, 128)).astype(np.float32))
    table = ccr.EmbeddingTable.from_tensor(P, device=torch.device("cuda:0"), exact=True)
    empty = _empty_set_mask(ccr, 5, 3000)
    got = table._search_exact(Q, 50, mask=empty, want_f64=True)
    ref = table._search_exact(Q, 50, want_f64=True)
    assert got[-1] == ref[-1] and (got[-1] == 5 or not fallback)
    _same(got[:-1], ref[:-1])
