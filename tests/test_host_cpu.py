"""CPU-only checks: the C-ABI library loads and exports every declared symbol, host-side logic
(lazy score algebra, fused-plan recognition, mask helpers, sharding arithmetic) behaves like the
reference.  No kernel is launched here."""
import ctypes
import operator
import os
import re

import numpy as np
import pytest
import scipy.sparse as sps
import torch

import cases
import _ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ccr_b200 import _lib

    header = open(os.path.join(ROOT, "include", "ccr_b200.h")).read()
    declared = set(re.findall(r"\b(ccr_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name
    assert _lib.lib().ccr_abi_version() == _lib.ABI_VERSION == 6


def test_planning_entry_points_work_without_gpu():
    from ccr_b200 import _lib

    L = _lib.lib()
    assert L.ccr_score_topk_workspace_bytes(4096, 8841823, 768, 100, 0, -1, 0) > 0
    assert L.ccr_score_topk_workspace_bytes(0, 100, 64, 5, 0, -1, 0) > 0        # B == 0 must not crash
    assert L.ccr_score_topk_workspace_bytes(4, 100, 63, 5, 0, -1, 0) == 0       # D % 8 != 0 -> invalid
    assert L.ccr_score_topk_workspace_bytes(4, 100, 64, 5000, 0, -1, 0) == 0    # k > CCR_MAX_K
    assert L.ccr_choose_algo(4, 1000, 768, 10) == _lib.ALGO_SIMT
    assert L.ccr_choose_algo(4, 8841823, 768, 100) == _lib.ALGO_TCGEN05
    assert L.ccr_choose_algo(512, 1000, 768, 10) == _lib.ALGO_TCGEN05
    info = _lib.plan_info(4096, 8841823, 768, 100)
    assert info["n_q_tiles"] == 16 and info["cand_capacity"] == 384 and info["n_splits"] >= 5  # 16 CTA-pair tiles
    assert info["two_cta"] == 1 and info["seed_items"] > 0 and info["n_kernel_launches"] == 4
    masked = _lib.plan_info(4096, 8841823, 768, 100, mask_nnz=30000, mask_max_row_nnz=64)
    assert masked["n_kernel_launches"] == 5 and masked["cand_capacity"] == 512  # + override kernel; k + 64 kept
    assert _lib.plan_info(384, 8841823, 768, 100)["n_q_tiles"] == 3  # odd tile count: single CTAs


def test_env_knobs_are_parsed_once_and_reloadable():
    from ccr_b200 import _lib

    from select_oracle import levers

    base = _lib.plan_info(512, 8841823, 768, 100)
    assert base["two_cta"] == 1
    with levers(_reload=False, CCR_2CTA="0"):
        assert _lib.plan_info(512, 8841823, 768, 100)["two_cta"] == 1   # cached knobs: no effect yet
        _lib.reload_env()
        assert _lib.plan_info(512, 8841823, 768, 100)["two_cta"] == 0
    assert _lib.plan_info(512, 8841823, 768, 100) == base


def test_product_refuses_cpu_tensors():
    import ccr_b200

    with pytest.raises(RuntimeError, match="CUDA"):
        ccr_b200.score_topk(torch.zeros(2, 8, dtype=torch.bfloat16), torch.zeros(4, 8, dtype=torch.bfloat16), 1)
    with pytest.raises(RuntimeError):
        ccr_b200.EmbeddingTable(10, 8, device="cpu")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "crowd-coachable-recommendations_b200", "ccr_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("al_oracle_agent", ""), fn


def test_shard_bounds_partition():
    from ccr_b200 import shard_bounds

    for n, g in [(10, 3), (8841823, 8), (5, 8), (0, 2), (100_000_000, 8)]:
        parts = [shard_bounds(n, g, r) for r in range(g)]
        assert parts[0][0] == 0 and parts[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
        assert all(hi - lo <= -(-n // g) for lo, hi in parts)


def test_fused_plan_recognition():
    import ccr_b200 as C

    c = cases.rime_case("mask_prior_k10")
    S = C.LazyDenseMatrix(c["U"]) @ C.LazyDenseMatrix(c["V"]).T
    plan = C.fused_plan(S)
    assert plan is not None and plan.sparse is None and plan.shape == (17, 257)
    S2 = S + c["prior"] - c["prior"] * 0.5
    plan2 = C.fused_plan(S2)
    assert plan2 is not None
    np.testing.assert_allclose(plan2.sparse.toarray(), (c["prior"] * 0.5).toarray())
    assert C.fused_plan(S.exp()) is None
    assert C.fused_plan(S * 2.0) is None
    assert C.fused_plan(C.LazyDenseMatrix(np.zeros((3, 4)))) is None
    # row slicing keeps the right factor object (so its device table is uploaded once)
    assert S2[0:4].children[0].children[0].right is S.right


@pytest.mark.skipif(not _ref_loader.reference_available(), reason="needs /root/reference")
def test_lazy_algebra_matches_reference_classes():
    import ccr_b200 as C

    ru = _ref_loader.load_rime_lite_util()
    c = cases.rime_case("mask_prior_k10")
    ours = C.LazyDenseMatrix(c["U"]) @ C.LazyDenseMatrix(c["V"]).T + c["prior"]
    ref = ru.LazyDenseMatrix(c["U"]) @ ru.LazyDenseMatrix(c["V"]).T + c["prior"]
    assert ours.shape == ref.shape and len(ours) == len(ref) and ours.size == ref.size
    assert ours.batch_size == ref.batch_size
    for key in (slice(0, 5), slice(3, 17), [1, 4, 9]):
        a, b = ours[key], ref[key]
        assert a.shape == b.shape
        torch.testing.assert_close(a.as_tensor("cpu"), b.as_tensor("cpu"))
    torch.testing.assert_close(ours.T.as_tensor("cpu"), ref.T.as_tensor("cpu"))
    parts_o = [ours[i:min(17, i + 4)] for i in range(0, 17, 4)]
    parts_r = [ref[i:min(17, i + 4)] for i in range(0, 17, 4)]
    torch.testing.assert_close(ours.collate_fn(parts_o).as_tensor("cpu"), ref.collate_fn(parts_r).as_tensor("cpu"))
    assert float(C.score_op(ours, "max")) == float(ru.score_op(ref, "max"))
    e_o, e_r = (ours * 0.5).sigmoid(), (ref * 0.5).sigmoid()
    torch.testing.assert_close(e_o.as_tensor("cpu"), e_r.as_tensor("cpu"))
    s_o, s_r = C.auto_cast_lazy_score(c["prior"]), ru.auto_cast_lazy_score(c["prior"])
    torch.testing.assert_close(s_o[2:6].as_tensor("cpu"), s_r[2:6].as_tensor("cpu"))
    rows_o, rows_r = [s_o[i] for i in range(3)], [s_r[i] for i in range(3)]
    torch.testing.assert_close(type(rows_o[0]).collate_fn(rows_o).as_tensor("cpu"),
                               type(rows_r[0]).collate_fn(rows_r).as_tensor("cpu"))


@pytest.mark.parametrize("name", list(cases.RIME_CASES))
def test_lazy_algebra_matches_stored_reference_output(name, golden_dir, monkeypatch):
    """Every operation test_lazy_algebra_matches_reference_classes compares, without the reference tree:
    the full matrix against the reference's stored output of the same expression (tests/golden/
    rime_<case>.npz: dtype, shape, head block), everything derived from it against the oracle's restatement
    of ``as_tensor`` (pinned to that stored output by test_oracle_golden.py)."""
    import ccr_b200 as C
    from oracle import ccr_oracle as O

    g = np.load(os.path.join(golden_dir, f"rime_{name}.npz"))
    c = cases.rime_case(name)
    S = C.LazyDenseMatrix(c["U"]) @ C.LazyDenseMatrix(c["V"]).T
    if c["prior"] is not None:
        S = S + c["prior"]
    ref = O.lazy_score_dense_ref(c["U"], c["V"], c["prior"])
    dense = S.as_tensor("cpu")
    assert str(dense.dtype) == str(g["dense_dtype"]) and tuple(dense.shape) == tuple(g["shape"])
    np.testing.assert_array_equal(dense[:4, :16].numpy().astype(np.float64), g["dense_head"])
    torch.testing.assert_close(dense, ref, rtol=0, atol=0)
    B, N = S.shape
    assert S.shape == tuple(ref.shape) and len(S) == B and S.size == B * N
    # the reference's row-batch heuristic (score_array.py:8-18), set small enough to stream several batches
    monkeypatch.setenv("BATCH_SIZE_FRAC", "1e-9")
    mem = torch.cuda.get_device_properties(0).total_memory if torch.cuda.device_count() else 16e9
    n_batches = int(B / (mem / 8 / N * 1e-9)) + 1
    assert S.batch_size == int(np.ceil(B / n_batches)) < B
    for key in (slice(0, 5), slice(3, B), [1, 4, B - 1]):
        assert S[key].shape == tuple(ref[key].shape)
        torch.testing.assert_close(S[key].as_tensor("cpu"), ref[key])
    torch.testing.assert_close(S.T.as_tensor("cpu"), ref.T)
    parts = [S[i:min(B, i + 4)] for i in range(0, B, 4)]
    torch.testing.assert_close(S.collate_fn(parts).as_tensor("cpu"), ref)
    b = S.batch_size
    prior_rows = (lambda i: c["prior"][i:i + b]) if c["prior"] is not None else (lambda i: None)
    want = max(float(O.lazy_score_dense_ref(c["U"][i:i + b], c["V"], prior_rows(i)).max()) for i in range(0, B, b))
    assert float(C.score_op(S, "max")) == want == pytest.approx(float(ref.max()), rel=1e-6)
    # values only: no stored reference output pins the dtype of a float32 matrix times a Python scalar
    torch.testing.assert_close((S * 0.5).sigmoid().as_tensor("cpu").double(), (ref * 0.5).sigmoid().double())
    if c["prior"] is not None:
        prior = torch.as_tensor(c["prior"].toarray())
        P = C.auto_cast_lazy_score(c["prior"])
        torch.testing.assert_close(P[2:6].as_tensor("cpu"), prior[2:6])
        rows = [P[i] for i in range(3)]
        torch.testing.assert_close(type(rows[0]).collate_fn(rows).as_tensor("cpu"), prior[:3])


def test_mask_helpers_on_cpu_arrays():
    """SparseMask canonicalisation / row slicing / column sharding arithmetic (host arrays only)."""
    from ccr_b200 import engine

    def host(m):  # build without touching a device
        return m

    class _M(engine.SparseMask):
        def __init__(self, indptr, cols, vals, n_cols, mode, device=None):
            self.n_rows = len(indptr) - 1
            self.n_cols = int(n_cols)
            self.mode = mode
            self.nnz = int(indptr[-1])
            self.host = (np.asarray(indptr, np.int64), np.asarray(cols, np.int32), np.asarray(vals, np.float64))
            self.max_row_nnz = int(np.diff(self.host[0]).max()) if self.n_rows else 0
            self.device = None

    engine_SparseMask = engine.SparseMask
    try:
        engine.SparseMask = _M
        m = _M([0, 2, 2, 5], [1, 7, 0, 4, 9], [-1.0, -2.0, 3.0, 4.0, 5.0], 10, engine.MASK_ADD)
        r = engine_SparseMask.rows(m, 1, 3)
        assert r.host[0].tolist() == [0, 0, 3] and r.host[1].tolist() == [0, 4, 9]
        s = engine_SparseMask.column_shard(m, 4, 10)
        assert s.n_cols == 6 and s.host[0].tolist() == [0, 1, 1, 3]
        assert s.host[1].tolist() == [3, 0, 5] and s.host[2].tolist() == [-2.0, 4.0, 5.0]
        e = engine_SparseMask.column_shard(m, 2, 4)
        assert e.nnz == 0 and e.host[0].tolist() == [0, 0, 0, 0]
    finally:
        engine.SparseMask = engine_SparseMask


def test_sparse_mask_from_flat_equals_from_lists(monkeypatch):
    """Vectorised block-mask construction (rows back to back, duplicates, empty rows) builds the
    same CSR as the per-row path; device upload stubbed out (host logic only)."""
    from ccr_b200 import engine

    monkeypatch.setattr(torch.Tensor, "to", lambda self, *a, **k: self)
    rs = np.random.RandomState(0)
    rows = [rs.randint(0, 50, size=rs.randint(0, 12)) for _ in range(40)] + [np.zeros(0, dtype=np.int64)]
    a = engine.SparseMask.from_lists(rows, 50, -1e6, engine.MASK_SET, "cpu")
    b = engine.SparseMask.from_flat([len(r) for r in rows], np.concatenate(rows), 50, -1e6, engine.MASK_SET, "cpu")
    for x, y in zip(a.host, b.host):
        np.testing.assert_array_equal(x, y)
    assert a.max_row_nnz == b.max_row_nnz and b.n_rows == 41
    with pytest.raises(IndexError):
        engine.SparseMask.from_flat([1], [50], 50, -1e6, engine.MASK_SET, "cpu")


def test_expression_recognition_factor_vs_materialised(monkeypatch):
    """Which expressions go to the fused kernel (factor pair), which to the dense top-k
    (materialised matrix), which are refused -- host-side logic only."""
    import scipy.sparse as sps

    import ccr_b200 as ccr

    U, V = np.ones((3, 8), np.float32), np.ones((5, 8), np.float32)
    prior = sps.csr_matrix(([1.0], ([0], [1])), shape=(3, 5))
    mm = ccr.LazyDenseMatrix(U) @ ccr.LazyDenseMatrix(V).T
    dense = ccr.LazyDenseMatrix(np.ones((3, 5), np.float32))
    assert ccr.fused_plan(mm) is not None and ccr.dense_plan(mm) is None
    assert ccr.fused_plan(mm + prior).sparse.nnz == 1 and ccr.fused_plan(mm - prior).sparse[0, 1] == -1.0
    assert ccr.fused_plan(dense) is None and ccr.dense_plan(dense) is not None
    p = ccr.dense_plan(dense + prior - prior * 2.0) if hasattr(prior, "__mul__") else None
    assert p is not None and p.sparse[0, 1] == -1.0 and p.shape == (3, 5)
    assert ccr.dense_plan(dense + dense) is None and ccr.fused_plan(mm + mm) is None   # two dense terms
    assert ccr.dense_plan(dense.exp()) is None and ccr.fused_plan(mm.exp()) is None    # non-linear
    assert ccr.dense_plan(ccr.auto_cast_lazy_score(np.zeros((2, 2)))) is not None      # plain ndarray
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)                       # also where a GPU is
    with pytest.raises(RuntimeError, match="CUDA"):                                      # no CPU path behind it
        ccr._assign_topk(dense, 2)


@pytest.mark.parametrize("sim", ["dot", "cos"])
def test_transform_scores_factor_pair_equals_reference_matrix(sim):
    """bbpr.py:528-550 as a lazy factor pair: its product is the reference's dense matrix."""
    import ccr_b200 as ccr
    from oracle import ccr_oracle as O

    rs = np.random.RandomState(4)
    all_emb = rs.standard_normal((60, 16)).astype(np.float32)
    i_to_ptr, j_to_ptr = rs.randint(0, 60, size=9), rs.permutation(60)[:41]
    S = ccr.transform_scores(all_emb, i_to_ptr, j_to_ptr, sim_type=sim)
    assert S.shape == (9, 41) and ccr.fused_plan(S) is not None
    want = O.transform_scores_ref(all_emb, i_to_ptr, j_to_ptr, 16, sim).numpy()
    np.testing.assert_allclose(S.left.c @ S.right.c, want, rtol=1e-5, atol=1e-5)
    assert ccr.fused_plan(S[2:5]).shape == (3, 41)  # row slicing keeps the factor form


def test_bench_reference_arm_contract(capsys, monkeypatch):
    """`bench.py --impl reference`: exactly --warmup + --steps steps of the CPU path, the product arm's
    `config` dict verbatim, the sample size bounded by a time budget (no GPU involved)."""
    import argparse
    import json

    import bench

    assert bench.reference_sample_queries(25, bench.N_ITEMS) == 7      # the driver's 20 + 5 steps
    assert bench.reference_sample_queries(13, bench.N_ITEMS) == 17     # bench.py's defaults
    assert bench.reference_sample_queries(2, bench.N_ITEMS) == 32      # capped
    assert bench.reference_sample_queries(10_000, bench.N_ITEMS) == 1  # never zero
    calls = []
    monkeypatch.setattr(bench, "cpu_reference_step", lambda P, n, seed=0: calls.append((n, seed)) or 0.01)
    monkeypatch.setattr(bench, "host_corpus", lambda n, seed=0: torch.zeros((4, bench.DIM)))
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    a = argparse.Namespace(gpus=1, steps=4, warmup=2, n_items=50_000, k=100, batch=4096, metric="m", workload="w")
    bench.run_reference(a)
    line = json.loads(capsys.readouterr().out)
    assert (line["impl"], line["steps"], line["warmup"]) == ("reference", 4, 2)
    assert len(calls) == 6 and len({n for n, _ in calls}) == 1 and calls[0][0] == line["sample_queries_per_step"]
    assert line["config"] == bench.workload_config(a, 1, 50_000)
    assert line["config"]["queries_per_step"] == 4096 and "plan" not in line["config"]
    assert line["e2e"] == {"value": line["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]


def test_bench_dump_outputs_and_steps_option(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 / float64 .npy files; above the size limit the same seeded row
    sample of every array plus its row numbers, identical from run to run.  `--steps` below 1 and a dump of the
    reference arm are refused."""
    import bench

    s = np.arange(40 * 3, dtype=np.float32).reshape(40, 3)
    i = s.astype(np.float64) * 2
    bench.dump_outputs(str(tmp_path / "all"), {"scores": s, "ids": i})
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "scores.npy"), s)
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "ids.npy"), i)
    assert not (tmp_path / "all" / "rows.npy").exists()
    limit = 10 * (3 * 4 + 3 * 8 + 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"scores": s, "ids": i}, limit=limit)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("scores", "ids", "rows")}
    rows = got["rows"].astype(np.int64)
    assert got["rows"].dtype == np.float64 and len(rows) == 10 and (np.diff(rows) > 0).all()
    assert sum(a.nbytes for a in got.values()) <= limit
    np.testing.assert_array_equal(got["scores"], s[rows])
    np.testing.assert_array_equal(got["ids"], i[rows])
    for n, a in got.items():
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f"{n}.npy"), a)
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "c"), {"ids": i.astype(np.int64)})
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "3", "--dump-outputs", str(tmp_path)])
    a = bench.parse()
    assert a.steps == 3 and a.dump_outputs == str(tmp_path)
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr("sys.argv", ["bench.py", *argv])
        with pytest.raises(SystemExit):
            bench.parse()
