"""Every launch plan of the fused score-and-rank path, bit-exact against the kernels' own scores
(select_oracle.py, DESIGN.md section 6): the tensor-core kernel must return exactly the top k of the dense
tile scores with the mask overrides applied, ids and float64 values identical, ties to the lowest id; the
CUDA-core kernel is held to a rigorous fp32 summation bound.  Each case pins one branch of the planner
(tests/test_select_oracle_cpu.py asserts that it reaches it) and runs bit-identically under the levers that
change scheduling only.  Needs a B200."""
import numpy as np
import pytest
import torch

import cases
import select_oracle as SO
from select_oracle import lever  # noqa: F401  (fixture)
from test_gpu_fullsize import N_MARCO, N_NQ, _queries, bench, big  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

SET, ADD = SO.MASK_SET, SO.MASK_ADD

# id, shape, operands, mask and the branch each case pins ("want": asserted on plan_info by the CPU test).
# mask: (mode, h) = random rows of 0..h entries; "big_row": one row with exactly that many entries;
# "bound": device CSR whose nnz / max_row_nnz are upper bounds (max_row_nnz -1 = unknown).
CASES = [
    dict(id="01-simt-auto", B=4, N=5000, D=64, k=10, algo=0,
         want=dict(algo=1)),
    dict(id="02-simt-forced-row-groups", B=300, N=30_000, D=768, k=1001, algo=1, mask=(SET, 40),
         want=dict(algo=1, n_q_tiles=38)),
    dict(id="03-single-one-unit-short-batch-qpitch", B=5, N=5000, D=72, k=100, algo=2, mask=(ADD, 40), q_pitch=80,
         want=dict(algo=2, two_cta=0, n_q_tiles=1, include=True, seeded=False)),
    dict(id="04-single-odd-tiles-inline-throttle-f16", B=384, N=20_000, D=128, k=10, algo=2, mask=(SET, 40), f16=True,
         want=dict(algo=2, two_cta=0, n_q_tiles=3, include=True, poller=False)),
    dict(id="05-one-pair-tile-item-pitch", B=256, N=5000, D=200, k=7, algo=2, i_pitch=256,
         want=dict(algo=2, two_cta=1, n_q_tiles=1, seeded=False)),
    dict(id="06-seed-hist-pairs-include-dups", B=512, N=300_000, D=64, k=100, algo=2, mask=(SET, 40), table="dup",
         keys=True, want=dict(algo=2, two_cta=1, include=True, seeded=True)),
    dict(id="07-include-at-h256", B=200, N=300_000, D=64, k=100, algo=2, mask=(ADD, 40), big_row=256,
         want=dict(algo=2, include=True, seeded=True)),
    dict(id="08-exclude-at-h257", B=200, N=300_000, D=64, k=100, algo=2, mask=(ADD, 40), big_row=257,
         want=dict(algo=2, include=False, seeded=True)),
    dict(id="09a-exclude-from-bounds", B=200, N=300_000, D=64, k=100, algo=2, mask=(SET, 40), bound=300,
         want=dict(algo=2, include=False, seeded=True)),
    dict(id="09b-exclude-unknown-h", B=200, N=300_000, D=64, k=100, algo=2, mask=(SET, 40), bound=-1,
         want=dict(algo=2, include=False, seeded=True)),
    dict(id="10a-k+h=2048-include", B=64, N=300_000, D=64, k=2000, algo=2, mask=(SET, 40), big_row=48, keys=True,
         want=dict(algo=2, include=True, seeded=True)),
    dict(id="10b-k+h=2049-exclude", B=64, N=300_000, D=64, k=2000, algo=2, mask=(SET, 40), big_row=49, keys=True,
         want=dict(algo=2, include=False, seeded=True)),
    dict(id="11-seed-at-floor-cos-f16", B=130, N=1 << 18, D=64, k=2048, algo=2, sim="cos", f16=True,
         want=dict(algo=2, two_cta=1, seeded=True, seed_items=16 * 2048)),
    dict(id="12a-unseeded-below-2^18", B=1, N=(1 << 18) - 1, D=64, k=1, algo=0,
         want=dict(algo=2, seeded=False)),
    dict(id="12b-seeded-at-2^18", B=1, N=1 << 18, D=64, k=1, algo=0,
         want=dict(algo=2, seeded=True)),
    dict(id="13-32-pair-tiles-poller", B=8192, N=270_000, D=64, k=10, algo=2,
         want=dict(algo=2, two_cta=1, n_q_tiles=32, poller=True)),
    dict(id="14-32-single-tiles-poller", B=4096, N=270_000, D=64, k=10, algo=2, mask=(SET, 40),
         levers=dict(CCR_2CTA="0"), want=dict(algo=2, two_cta=0, n_q_tiles=32, poller=True)),
    dict(id="15-B8193-single-padded", B=8193, N=270_000, D=64, k=10, algo=2, mask=(ADD, 40),
         want=dict(algo=2, two_cta=0, n_q_tiles=65, poller=True)),
    dict(id="16-50-distinct-rows-single-ctas", B=1100, N=300_000, D=64, k=1001, algo=2, mask=(SET, 40),
         table="distinct50", keys=True, want=dict(algo=2, two_cta=0, n_q_tiles=9, include=True, seeded=True)),
    dict(id="17-all-scores-tie", B=150, N=300_000, D=64, k=2048, algo=2, table="same",
         want=dict(algo=2, two_cta=1, seeded=True)),
    dict(id="18-D4096", B=130, N=20_000, D=4096, k=10, algo=2,
         want=dict(algo=2, two_cta=1)),
    dict(id="19-D8-k=N", B=9, N=33, D=8, k=33, algo=0, mask=(ADD, 10),
         want=dict(algo=2, n_q_tiles=1, include=True)),
    dict(id="20-k>N-allow-short-id-offset", B=7, N=100, D=64, k=300, algo=2, mask=(SET, 40), allow_short=True,
         id_offset=(1 << 31) + 5, want=dict(algo=2, include=True)),
]


def case_seed(c):
    return sum(map(ord, c["id"])) * 7 + c["B"]


def _distinct(rs, N, n):
    """n distinct sorted ids below N (rejection sampling: rs.choice permutes all N per row)."""
    if N < 10 * n + 100:
        return np.sort(rs.choice(N, size=n, replace=False))
    u = rs.randint(0, N, size=n + 16)
    _, first = np.unique(u, return_index=True)
    u = u[np.sort(first)][:n]
    assert len(u) == n
    return np.sort(u)


_MASKS = {}


def case_mask(c):
    """Host CSR (indptr int64, cols int32, vals float64, mode) of a case, or None."""
    if "mask" not in c:
        return None
    if c["id"] in _MASKS:
        return _MASKS[c["id"]]
    mode, h = c["mask"]
    B, N = c["B"], c["N"]
    rs = np.random.RandomState(case_seed(c))
    sizes = rs.randint(0, min(N, h) + 1, size=B)
    if "big_row" in c:
        sizes[rs.randint(B)] = c["big_row"]
    cols = [_distinct(rs, N, n) for n in sizes]
    indptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    cols = np.concatenate(cols).astype(np.int32)
    if mode == SET:
        vals = np.full(len(cols), -1e6)
    else:  # blocks, dominating priors, and priors that interleave with the scores
        vals = np.where(rs.rand(len(cols)) < 0.3, -1e10,
                        np.where(rs.rand(len(cols)) < 0.5, 1e5, rs.standard_normal(len(cols)) * 3))
    _MASKS[c["id"]] = (indptr, cols, vals, mode)
    return _MASKS[c["id"]]


def mask_args(c, host):
    """(nnz, max_row_nnz) the call passes for the case's mask."""
    if host is None:
        return 0, -1
    nnz = int(host[0][-1])
    if "bound" in c:
        return nnz + 1000, c["bound"]
    return nnz, int(np.diff(host[0]).max())


def case_flags(c):
    from ccr_b200 import _lib

    return (c["algo"] | (_lib.FLAG_F16 if c.get("f16") else 0) | (_lib.FLAG_ALLOW_SHORT if c.get("allow_short") else 0))


def plan_of(c, host=None):
    from ccr_b200 import _lib

    nnz, h = mask_args(c, host if host is not None else case_mask(c))
    return _lib.plan_info(c["B"], c["N"], c["D"], c["k"], flags=case_flags(c), mask_nnz=nnz, mask_max_row_nnz=h)


def variants(c, plan):
    """Levers that change scheduling only, where the plan uses what they change."""
    out = []
    if plan["algo"] != 2:
        return out
    if plan["n_q_tiles"] > 1:
        out += [dict(CCR_LEAD="2"), dict(CCR_LEAD="4")]
    if plan["seed_items"] > 0:
        out.append(dict(CCR_NO_HIST="1"))
    if c["B"] > 128:
        out.append(dict(CCR_2CTA="0" if plan["two_cta"] else "1"))
    return out


def _table_rows(c):
    N, D = c["N"], c["D"]
    rs = np.random.RandomState(case_seed(c) + 1)
    kind = c.get("table", "clustered" if c.get("sim") == "cos" else "randn")
    if kind == "same":
        return np.tile(rs.standard_normal((1, D)).astype(np.float32), (N, 1))
    if kind == "distinct50":
        return rs.standard_normal((50, D)).astype(np.float32)[rs.randint(0, 50, size=N)]
    P = cases.embeddings(case_seed(c) + 2, N, D, clustered=(kind == "clustered"))
    if kind == "dup":
        P[rs.randint(0, N, size=N // 4)] = P[rs.randint(0, N, size=N // 4)]
    return P


def _pitched(t, pitch):
    """``t`` [n, D] as a column slice of a NaN-padded [n, pitch] tensor (the kernels must never read past D)."""
    wide = torch.full((t.shape[0], pitch), float("nan"), dtype=t.dtype, device=t.device)
    wide[:, : t.shape[1]] = t
    return wide[:, : t.shape[1]]


def build(ccr, c):
    dev = torch.device("cuda:0")
    dtype = torch.float16 if c.get("f16") else torch.bfloat16
    cos = c.get("sim") == "cos"
    table = ccr.EmbeddingTable.from_tensor(torch.as_tensor(_table_rows(c)), device=dev, normalize=cos, dtype=dtype)
    assert table.ld == c["D"]
    q = table.encode_queries(torch.as_tensor(cases.embeddings(case_seed(c) + 3, c["B"], c["D"], clustered=cos)))
    items = table.data[: c["N"]]
    if "q_pitch" in c:
        q = _pitched(q, c["q_pitch"])
    if "i_pitch" in c:
        items = _pitched(items, c["i_pitch"])
    host = case_mask(c)
    mask = None
    if host is not None:
        ip, cols, vals, mode = host
        if "bound" in c:
            nnz, h = mask_args(c, host)
            pad = nnz - len(cols)  # room up to the bound, holding entries no kernel may read
            t_ip = torch.as_tensor(ip, device=dev)
            t_c = torch.as_tensor(np.concatenate([cols, np.zeros(pad, np.int32)]), device=dev)
            t_v = torch.as_tensor(np.concatenate([vals, np.full(pad, 1e30)]), device=dev)
            mask = ccr.SparseMask.from_device_tensors(t_ip, t_c, t_v, None, c["N"], mode, nnz=nnz, max_row_nnz=h)
        else:
            mask = ccr.SparseMask(ip, cols, vals, c["N"], mode, dev)
    return table, q, items, mask, host


def search(ccr, c, q, items, mask, **kw):
    return ccr.engine.score_topk(q, items, c["k"], mask=mask, id_offset=c.get("id_offset", 0), algo=c["algo"],
                                 allow_short=c.get("allow_short", False), n_items=c["N"], D=c["D"], **kw)


def same_bits(a, b):
    return all(torch.equal(x.view(torch.int64) if x.dtype == torch.float64 else
                           x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int64) if y.dtype == torch.float64 else
                           y.view(torch.int32) if y.dtype == torch.float32 else y) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def ccr():
    import ccr_b200

    assert torch.cuda.is_available()
    return ccr_b200


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_plan_matrix_exact(ccr, c, lever):
    lever(**c.get("levers", {}))
    table, q, items, mask, host = build(ccr, c)
    plan = plan_of(c, host)
    s, i, d = search(ccr, c, q, items, mask, want_f64=True)
    torch.cuda.synchronize()
    if plan["algo"] == 1:
        errs = SO.check_bounded(s.cpu().numpy(), i.cpu().numpy(), d.cpu().numpy(), q, items, c["D"], c["k"], host,
                                id_offset=c.get("id_offset", 0))
    else:
        want_v, want_i = SO.exact_reference(q, items, c["D"], c["k"], host, id_offset=c.get("id_offset", 0),
                                            allow_short=c.get("allow_short", False))
        errs = SO.check_exact(s.cpu().numpy(), i.cpu().numpy(), d.cpu().numpy(), want_v, want_i)
    assert not errs, errs
    for kv in variants(c, plan):
        with SO.levers(**kv):
            again = search(ccr, c, q, items, mask, want_f64=True)
        assert same_bits((s, i, d), again), kv
    if c.get("keys"):
        s2, i2, keys = search(ccr, c, q, items, mask, want_keys=True)
        assert same_bits((s, i), (s2, i2))
        us, ui = ccr.engine.unpack_topk_keys(keys)
        assert same_bits((s, i), (us, ui))


def _check_rows(ccr, table, q, N, k, mask):
    s, i, d = ccr.score_topk(q, table.data, k, mask=mask, n_items=N, D=table.ld, want_f64=True)
    torch.cuda.synchronize()
    want_v, want_i = SO.exact_reference(q, table.data, table.ld, k, mask, n_items=N)
    errs = SO.check_exact(s.cpu().numpy(), i.cpu().numpy(), d.cpu().numpy(), want_v, want_i)
    assert not errs, errs


def test_bench_workload_exact_every_row(ccr, bench, big):
    """bench.py's step (8,841,823 x 768, B = 4096, top-100, history mask): every row identical to the exact
    top k of the kernel's own scores."""
    B, k = 4096, bench.TOPK
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N_MARCO))
    mask = ccr.SparseMask(indptr, cols, vals, N_MARCO, ccr.MASK_SET, big.device)
    _check_rows(ccr, big, _queries(big, B), N_MARCO, k, mask)


def test_nq_shape_k1001_exact_every_row(ccr, bench, big):
    """The NQ shape as ranking() asks for it (2,681,468 x 768, k = 1001), with and without a block list."""
    B, k = 3452, 1001
    q = _queries(big, B, seed=11)
    indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, N_NQ, seed=5))
    mask = ccr.SparseMask(indptr, cols, vals, N_NQ, ccr.MASK_SET, big.device)
    _check_rows(ccr, big, q, N_NQ, k, mask)
    _check_rows(ccr, big, q[:700], N_NQ, k, None)
