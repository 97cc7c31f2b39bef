"""The workspace every top-k entry point asks for matches its size query.

Each entry is called with consistent arguments and a null workspace: it must return CCR_EWORKSPACE before any
device work, naming the bytes it needs.  The pointers are aligned dummies that are never dereferenced.  Without a
GPU the plans use the library's default SM count, the same in the entry and in its size query."""
import itertools
import re

import pytest
import torch

from ccr_b200 import _lib

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="checks the host side only, without a device")

P = 1 << 12  # aligned, never dereferenced
D = 768
SHAPES = [(B, N, k) for B, N, k in itertools.product([1, 100, 300, 4096], [1000, 300000, 8841823], [10, 100, 1001])
          if k <= N]
MASKS = [(0, -1)] + list(itertools.product([5000], [-1, 0, 3, 300]))


def _required(rc):
    """Bytes a call that returned CCR_EWORKSPACE says it needs."""
    msg = _lib.lib().ccr_last_error_string().decode()
    assert rc == _lib.EWORKSPACE, (rc, msg)
    m = re.fullmatch(r"workspace 0 < (\d+)", msg)
    assert m, msg
    return int(m.group(1))


@pytest.mark.parametrize("flags", [0, _lib.FLAG_F16, _lib.ALGO_SIMT])
@pytest.mark.parametrize("mode", [_lib.MASK_SET, _lib.MASK_ADD])
def test_fused_and_exact_need_what_the_size_query_says(mode, flags):
    L = _lib.lib()
    for (B, N, k), (nnz, h) in itertools.product(SHAPES, MASKS):
        rc = L.ccr_score_topk_bf16(P, B, D, P, N, D, D, k, P, P, P, nnz, h, mode, 0, P, P, P, None, 0, flags, None)
        assert _required(rc) == L.ccr_score_topk_workspace_bytes(B, N, D, k, nnz, h, flags), (B, N, k, nnz, h)
        rc = L.ccr_score_topk_exact(P, P, B, D, P, P, N, D, D, k, P, P, P, P, nnz, h, mode, 0, P, P, P, P, P, P, None, 0,
                                    flags, None)
        assert _required(rc) == L.ccr_score_topk_exact_workspace_bytes(B, N, D, k, nnz, h, flags), (B, N, k, nnz, h)


@pytest.mark.parametrize("mode", [_lib.MASK_SET, _lib.MASK_ADD])
def test_rerank_needs_what_the_size_query_says(mode):
    L = _lib.lib()
    for (B, N, k), nnz in itertools.product(SHAPES, [0, 5000]):
        cand_nnz = B * k
        rc = L.ccr_rerank_exact(P, B, D, P, N, D, D, k, P, P, cand_nnz, P, P, P, nnz, mode, 0, P, P, P, None, 0, 0,
                                None)
        assert _required(rc) == L.ccr_rerank_exact_workspace_bytes(B, cand_nnz, nnz), (B, N, k, nnz)


@pytest.mark.parametrize("mode", [_lib.MASK_SET, _lib.MASK_ADD])
def test_dense_topk_needs_what_the_size_query_says(mode):
    L = _lib.lib()
    for (B, N, k), (nnz, h) in itertools.product(SHAPES, MASKS):
        if nnz > 0 and h < 0:
            continue  # a mask without a row bound: see the test below
        rc = L.ccr_topk_dense_f32(P, B, N, N, k, P, P, P, nnz, h, mode, P, P, P, None, 0, None)
        size = L.ccr_topk_dense_workspace_bytes(B, N, k, nnz, h)
        if k + max(h, 0) > _lib.MAX_K:
            assert rc == _lib.EUNSUPPORTED and size == 0
        else:
            assert _required(rc) == size, (B, N, k, nnz, h)


def test_bm25_needs_at_most_what_the_size_query_says():
    L = _lib.lib()
    for (B, N, k), max_terms in itertools.product(SHAPES, [5, 32, 33, 500]):
        rc = L.ccr_bm25_topk(P, P, P, None, None, P, P, max_terms, B, N, k, P, P, None, 0, None)
        assert _required(rc) <= L.ccr_bm25_topk_workspace_bytes(B, N, k), (B, N, k, max_terms)


def test_dense_topk_mask_without_row_bound_says_so():
    L = _lib.lib()
    rc = L.ccr_topk_dense_f32(P, 4, 1000, 1000, 100, P, P, P, 5000, -1, _lib.MASK_SET, P, P, P, None, 0, None)
    assert rc == _lib.EUNSUPPORTED
    assert "mask_max_row_nnz" in L.ccr_last_error_string().decode()
    assert L.ccr_topk_dense_workspace_bytes(4, 1000, 100, 5000, -1) == 0
