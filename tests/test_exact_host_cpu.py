"""Exact fp32 ranking without a GPU: defaults, the k' rule and the error bound (DESIGN.md section 6b)."""
import inspect

import numpy as np
import pytest
import torch


def test_exact_defaults_to_false_and_reference_signatures_unchanged():
    import importlib

    al_rank, ranking, table = (importlib.import_module(f"ccr_b200.{m}") for m in ("al_rank", "ranking", "table"))

    util, metrics, dist = (importlib.import_module(f"ccr_b200.{m}") for m in ("util", "metrics", "dist"))
    for fn in (table.EmbeddingTable.__init__, table.EmbeddingTable.from_tensor, ranking.ranking,
               ranking.generate_embeddings_device, al_rank.rank_step, util._assign_topk, util.topk_lazy,
               metrics.evaluate_item_rec, dist.ShardedIndex.__init__, ranking.ranking_sharded):
        assert inspect.signature(fn).parameters["exact"].default is False, fn
    # the reference's positional parameters come first, as before
    assert list(inspect.signature(ranking.ranking).parameters)[:5] == [
        "corpus", "queries", "embedding_func", "batch_size", "block_dict"]
    assert list(inspect.signature(util._assign_topk).parameters)[:5] == ["S", "k", "tie_breaker", "device",
                                                                         "batch_size"]
    assert list(inspect.signature(metrics.evaluate_item_rec).parameters)[:4] == ["target_csr", "score_mat", "topk",
                                                                                "device"]


@pytest.mark.parametrize("exact", [True, False])
def test_rank_step_hands_exact_to_ranking(exact, tmp_path, monkeypatch):
    import importlib

    al_rank, ranking = (importlib.import_module(f"ccr_b200.{m}") for m in ("al_rank", "ranking"))
    seen = {}

    class Stop(Exception):
        pass

    def fake_ranking(*args, **kw):
        seen.update(kw)
        raise Stop

    monkeypatch.setattr(ranking, "ranking", fake_ranking)
    with pytest.raises(Stop):
        al_rank.rank_step({}, {}, {}, None, str(tmp_path), 0, {}, [], exact=exact)
    assert seen["exact"] is exact


@pytest.mark.parametrize("flags", [0, 0x40])
def test_k_candidates_rule(flags):
    from ccr_b200 import _lib

    for n in (1, 40, 1000, 20000, 8841823):
        for k in (1, 5, 40, 100, 1001, 2048):
            if k > n:
                continue
            kc = _lib.exact_k_candidates(4096, n, 768, k, flags)
            assert k <= kc <= min(n, _lib.MAX_K), (n, k, kc)


def test_bound_mirror_matches_library():
    from ccr_b200 import _lib, engine

    L = _lib.lib()
    for qn, v, D, f16 in ((1.0, 1.0, 768, 0), (27.7, 28.1, 768, 1), (1e-30, 3.0, 64, 1), (5e3, 1e4, 4096, 0)):
        assert engine.exact_error_bound(qn, v, D, f16) == L.ccr_exact_error_bound(qn, v, D, 0x40 if f16 else 0)


def _scan_emulation(Q, P, f16, rs, block):
    """Scan scores as the kernels compute them: operands rounded to the scan format, fp32 products summed
    in fp32 in blocks of ``block`` (random partial-sum order), blocks then summed in fp32."""
    if f16:
        q, p = Q.astype(np.float16).astype(np.float32), P.astype(np.float16).astype(np.float32)
    else:
        q = torch.as_tensor(Q).bfloat16().float().numpy()
        p = torch.as_tensor(P).bfloat16().float().numpy()
    prod = (q[:, None, :] * p[None, :, :]).astype(np.float32)  # exact: 16 / 22 significant bits
    D = Q.shape[1]
    perm = rs.permutation(D)
    prod = prod[:, :, perm]
    acc = np.zeros(prod.shape[:2], dtype=np.float32)
    for b0 in range(0, D, block):
        part = np.zeros(prod.shape[:2], dtype=np.float32)
        for d in range(b0, min(D, b0 + block)):
            part = (part + prod[:, :, d]).astype(np.float32)
        acc = (acc + part).astype(np.float32)
    return acc


@pytest.mark.parametrize("f16", [False, True])
def test_emulated_scan_stays_within_bound(f16):
    from ccr_b200 import engine

    rs = np.random.RandomState(1 + f16)
    worst = 0.0
    for trial in range(24):
        D = int(rs.choice([64, 128, 256, 768]))
        kind = trial % 4
        P = rs.standard_normal((40, D)).astype(np.float32)
        Q = rs.standard_normal((6, D)).astype(np.float32)
        if kind == 1:  # wide dynamic range
            P *= (10.0 ** rs.uniform(-3, 3, (40, 1))).astype(np.float32)
        elif kind == 2:  # heavy cancellation
            P[:, D // 2:] = -P[:, : D // 2] + (rs.standard_normal((40, D // 2)) * 1e-4).astype(np.float32)
            Q[:, D // 2:] = Q[:, : D // 2]
        elif kind == 3:  # near fp16's subnormal range
            P *= np.float32(2e-6)
        s_hat = _scan_emulation(Q, P, f16, rs, int(rs.choice([1, 8, 32, 128])))
        exact = (Q.astype(np.float64) @ P.astype(np.float64).T).astype(np.float32).astype(np.float64)
        qn = np.sqrt((Q.astype(np.float64) ** 2).sum(1))
        v = float(np.sqrt((P.astype(np.float64) ** 2).sum(1)).max())
        E = engine.exact_error_bound(qn, v, D, f16)
        ratio = np.abs(s_hat - exact) / E[:, None]
        worst = max(worst, float(ratio.max()))
    print(f"f16={f16}: max emulated |s^ - s| / E_row = {worst:.4f}")
    assert worst <= 1.0
