"""fp16 tables without a GPU: ABI flag and planning invariance, defaults, dtype checks, and the fp16
oracle against the reference's own GPU goldens."""
import importlib
import inspect
import itertools
import os
import re

import numpy as np
import pytest
import torch

import cases
import f16_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flag_f16_matches_header():
    from ccr_b200 import _lib

    header = open(os.path.join(ROOT, "include", "ccr_b200.h")).read()
    m = re.search(r"#define\s+CCR_FLAG_F16\s+(0x[0-9a-fA-F]+)", header)
    assert m and int(m.group(1), 16) == _lib.FLAG_F16
    # it must not collide with the algorithm bits or another flag
    assert _lib.FLAG_F16 & 0xF == 0  # CCR_ALGO_MASK
    assert _lib.FLAG_F16 not in (_lib.FLAG_ALLOW_SHORT, _lib.FLAG_PACKED_KEYS)


def test_plan_and_workspace_do_not_depend_on_f16():
    """Same 2 bytes per element: every launch parameter and the workspace size are those of bf16."""
    import ctypes

    from ccr_b200 import _lib

    L = _lib.lib()
    masks = [(0, -1), (4096 * 9, 40), (4096 * 300, 300)]  # none, include mode (h <= 256), exclude mode
    n = 0
    for B, N, k, (nnz, h), algo in itertools.product([0, 1, 8, 128, 384, 512, 4096, 8192, 16384],
                                                     [1000, 65535, 300000, 8841823], [1, 100, 1001, 2048],
                                                     masks, [0, 1, 2]):
        for extra in (0, _lib.FLAG_ALLOW_SHORT):
            flags = algo | extra
            a = (ctypes.c_int32 * 8)()
            b = (ctypes.c_int32 * 8)()
            ra = L.ccr_plan_info(B, N, 768, k, nnz, h, flags, a)
            rb = L.ccr_plan_info(B, N, 768, k, nnz, h, flags | _lib.FLAG_F16, b)
            assert ra == rb and list(a) == list(b), (B, N, k, nnz, h, flags)
            wa = L.ccr_score_topk_workspace_bytes(B, N, 768, k, nnz, h, flags)
            wb = L.ccr_score_topk_workspace_bytes(B, N, 768, k, nnz, h, flags | _lib.FLAG_F16)
            assert wa == wb, (B, N, k, nnz, h, flags)
            n += 1
    assert n == 9 * 4 * 4 * 3 * 3 * 2


@pytest.mark.parametrize("name", list(cases.CUDA_RANKING_CASES))
def test_fp16_oracle_reproduces_reference_gpu_golden(name, golden_dir):
    """Operands rounded to fp16 (the reference's autocast format) reproduce the reference's own B200
    ranking up to accumulation order; bf16 operands do not."""
    g = np.load(os.path.join(golden_dir, f"ranking_cuda_autocast_{name}.npz"))
    c = cases.ranking_case(name)
    k = g["order"].shape[1]
    v16, o16 = f16_ref.emulate_ranking(c, lambda x: x.half().float(), k)
    vbf, obf = f16_ref.emulate_ranking(c, lambda x: x.to(torch.bfloat16).float(), k)
    eq16, tie16, top16 = f16_ref.golden_agreement(v16, o16, g["scores"], g["order"])
    eqbf, tiebf, topbf = f16_ref.golden_agreement(vbf, obf, g["scores"], g["order"])
    print(f"{name}: fp16 score-equal {eq16:.4f} tie-aware {tie16:.4f} top2 {top16:.3f} | "
          f"bf16 {eqbf:.4f} {tiebf:.4f} {topbf:.3f}")
    assert eq16 >= 0.995 and tie16 >= 0.995, (eq16, tie16)
    assert eq16 > eqbf and tie16 > tiebf


def test_oracle_f16_wrappers_round_where_the_oracle_does():
    from oracle import ccr_oracle as O

    rs = np.random.RandomState(0)
    Q, P = rs.standard_normal((5, 64)).astype(np.float32), rs.standard_normal((300, 64)).astype(np.float32)
    for sim in ("dot", "cos"):
        full = f16_ref.full_scores_ref_f16(Q, P, sim=sim)
        Qh, Ph = torch.as_tensor(Q), torch.as_tensor(P)
        if sim == "cos":
            Qh, Ph = O.normalize_rows_ref(Qh), O.normalize_rows_ref(Ph)
        torch.testing.assert_close(full, Qh.half().float() @ Ph.half().float().T, rtol=0, atol=0)
        s, i = f16_ref.score_topk_ref_f16(Q, P, 7, sim=sim)
        want = torch.sort(full, dim=1, descending=True, stable=True)
        assert torch.equal(i, want.indices[:, :7]) and torch.equal(s, want.values[:, :7])
        # and it differs from the bf16 default
        assert not torch.equal(full, O.full_scores_ref(Q, P, sim=sim))


def test_defaults_are_bf16_and_bad_dtypes_raise():
    import ccr_b200
    from ccr_b200 import al_rank, dist, table

    ranking_mod = importlib.import_module("ccr_b200.ranking")  # the package attribute `ranking` is the function
    sig = inspect.signature
    assert sig(table.EmbeddingTable).parameters["dtype"].default is torch.bfloat16
    assert sig(table.EmbeddingTable.from_tensor).parameters["dtype"].default is torch.bfloat16
    assert sig(dist.ShardedIndex).parameters["dtype"].default is torch.bfloat16
    assert sig(ranking_mod.ranking).parameters["table_dtype"].default is torch.bfloat16
    assert sig(ranking_mod.ranking_sharded).parameters["table_dtype"].default is torch.bfloat16
    assert sig(ranking_mod.generate_embeddings_device).parameters["dtype"].default is torch.bfloat16
    assert sig(al_rank.rank_step).parameters["table_dtype"].default is torch.bfloat16
    # the reference-facing positional signature is unchanged
    assert list(sig(ranking_mod.ranking).parameters)[:5] == ["corpus", "queries", "embedding_func", "batch_size",
                                                             "block_dict"]
    for bad in (torch.float32, torch.float64, torch.int8):
        with pytest.raises(ValueError, match="dtype"):
            ccr_b200.EmbeddingTable(4, 64, device="cpu", dtype=bad)  # checked before the device
        with pytest.raises(ValueError, match="dtype"):
            ranking_mod.ranking({}, {}, None, 1, table_dtype=bad)
    # a valid dtype still refuses a CPU table
    with pytest.raises(RuntimeError, match="CUDA"):
        ccr_b200.EmbeddingTable(4, 64, device="cpu", dtype=torch.float16)


def test_mixed_operand_dtypes_raise_type_error():
    from ccr_b200 import engine

    a = torch.zeros(2, 8, dtype=torch.float16)
    b = torch.zeros(3, 8, dtype=torch.bfloat16)
    for q, p in ((a, b), (b, a), (a.float(), a)):
        with pytest.raises(TypeError):
            engine._operand_f16(q, p)
    assert engine._operand_f16(a, a) is True and engine._operand_f16(b, b) is False
