"""Randomised small-shape parity sweep through the C ABI against the CPU oracle: tile-boundary
batch / corpus sizes, odd dims, k up to N, light and heavy masks (include and exclude modes),
SET and ADD (positive priors), dot and cos, bf16 and fp16 tables, both kernels, 1-CTA and 2-CTA tensor-core
variants; besides the tolerance rule, every case is checked bit-exactly (tensor-core kernel) or against the fp32
summation bound (CUDA-core kernel) by select_oracle."""
import numpy as np
import pytest
import torch

import cases
import f16_ref
import select_oracle as SO
from oracle import ccr_oracle as O
from select_oracle import lever  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def _one_case(ccr, rs, B, N, D, k, mode, heavy, sim, algo, dtype):
    dev = torch.device("cuda:0")
    P = cases.embeddings(int(rs.randint(1 << 30)), N, D, clustered=(sim == "cos"))
    Q = cases.embeddings(int(rs.randint(1 << 30)), B, D, clustered=(sim == "cos"))
    if rs.rand() < 0.3:  # exact ties: duplicate some items
        P[rs.randint(0, N, size=N // 4)] = P[rs.randint(0, N, size=N // 4)]
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(P), device=dev, normalize=(sim == "cos"), dtype=dtype)
    mask = None
    if mode != O.MASK_NONE:
        hi = min(N, 600 if heavy else 40)
        rows = [rs.choice(N, size=rs.randint(0, hi + 1), replace=False) for _ in range(B)]
        if mode == O.MASK_SET:
            mask = ccr.SparseMask.from_lists(rows, N, -1e6, ccr.MASK_SET, dev)
        else:
            indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
            cols = np.concatenate([np.sort(r) for r in rows]) if B else np.zeros(0)
            vals = np.where(rs.rand(len(cols)) < 0.5, -1e10, rs.choice([1.0, 1e5], size=len(cols)))
            mask = ccr.SparseMask(indptr, cols, vals, N, ccr.MASK_ADD, dev)
    q = table.encode_queries(torch.as_tensor(Q))
    s, i, d = table.search(q, k, mask=mask, algo=algo, want_f64=True, encoded=True)
    torch.cuda.synchronize()
    errs = SO.check_kernel(algo, s, i, d, q, table.data, table.ld, k, mask, n_items=N)
    if errs:
        return errs
    ref = f16_ref.full_scores_ref_f16 if dtype == torch.float16 else O.full_scores_ref
    full = ref(Q, P, mask=mask.host if mask else None, mode=mode, sim=sim).numpy()
    # cos: the fp32 norm is summed in a different order than torch's, so a normalised element can land
    # on the other side of a bf16 rounding boundary (1 bf16 ulp of one factor) -> absolute slack on the
    # unit-scale cos scores; dot: the bf16 inputs are bit-identical, only fp32 summation order differs
    live = np.abs(full[np.abs(full) < 1e5])
    atol = 2e-3 if sim == "cos" else 1e-5 * float(live.max() if live.size else 1.0)
    return O.check_topk(d.cpu().numpy(), i.cpu().numpy(), full_scores=full, rtol=1e-2, atol=atol)


@pytest.mark.parametrize("seed", range(6))
def test_fuzz_against_oracle(seed, lever):
    import ccr_b200 as ccr

    rs = np.random.RandomState(1000 + seed)
    Bs = [1, 2, 7, 8, 9, 64, 127, 128, 129, 200, 255, 256, 257, 384, 385, 400]
    Ns = [1, 2, 31, 32, 33, 255, 256, 257, 511, 512, 513, 1000, 2049, 5000]
    Ds = [8, 24, 64, 72, 128, 200, 768]
    for it in range(14):
        B, N, D = int(rs.choice(Bs)), int(rs.choice(Ns)), int(rs.choice(Ds))
        k = int(min(N, 2048, rs.choice([1, 2, 5, 10, 100, 300, 1001, N])))
        mode = int(rs.choice([O.MASK_NONE, O.MASK_SET, O.MASK_ADD]))
        heavy = bool(rs.rand() < 0.3)
        sim = "cos" if rs.rand() < 0.25 else "dot"
        algo = int(rs.choice([1, 2, 2]))
        two = str(int(rs.rand() < 0.5))
        dtype = torch.float16 if rs.rand() < 0.5 else torch.bfloat16
        lever(CCR_2CTA=two)
        errs = _one_case(ccr, rs, B, N, D, k, mode, heavy, sim, algo, dtype)
        assert not errs, (dict(B=B, N=N, D=D, k=k, mode=mode, heavy=heavy, sim=sim, algo=algo, two_cta=two,
                               dtype=dtype), errs[:3])
