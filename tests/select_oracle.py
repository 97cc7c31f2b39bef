"""Exact oracle for the selection half of the fused score-and-rank path (DESIGN.md section 6).

The only inexact step of the tensor-core path is the fp32 accumulation inside the MMA, and it need not be
modelled: ``ccr_score_dense_f32`` / ``_f16`` on tiles of >= 2^20 scores run ``select_tc_kernel`` with the same
K loop, instruction descriptor and TMA boxes as the fused kernel and only a store epilogue, so every (row,
item) score they write is the fused kernel's score, bit for bit.  Masked items take the value the override
kernel computes, which is emulated here exactly (SET: the value; ADD: a fixed fp32 lane / butterfly order
plus the value in float64).  Ranking those values by the kernels' total order -- ``ord64(value)``
descending, then id ascending, so -0.0 ranks just below +0.0 -- gives the exact top k of every launch plan.

The CUDA-core (SIMT) kernel sums in an order that depends on the item's slot in the warp; it is checked
against a rigorous bound instead (``check_bounded``).

Also the one way the tests set the library's CCR_* levers (``lever``): the library parses them once per
process, so a lever only takes effect through ``_lib.reload_env()``."""
import contextlib
import os

import numpy as np
import pytest
import torch

MASK_NONE, MASK_SET, MASK_ADD = 0, 1, 2
LEVERS = ("CCR_2CTA", "CCR_LEAD", "CCR_NO_HIST", "CCR_BM25_BLOCKWIDE", "CCR_EXACT_FALLBACK")
BLOCK_BYTES = 2 << 30   # fp32 scores per dense-tile call
DENSE_TC_MIN = 1 << 20  # ccr_score_dense takes the tensor-core path from this many scores (and >= 256 items)
ITEM_TILE = 256

# ---- levers ----

def _set_env(kv, reload=True):
    from ccr_b200 import _lib

    for key, v in kv.items():
        if key not in LEVERS:
            raise KeyError(f"{key} is not a CCR_* lever")
        if v is None:
            os.environ.pop(key, None)
        else:
            os.environ[key] = str(v)
    if reload:
        _lib.reload_env()


@contextlib.contextmanager
def levers(_reload=True, **kv):
    """Set CCR_* levers (None unsets one) for the body and make the library re-read them; on exit the old
    environment is restored and re-read.  ``_reload=False`` leaves the library's cached copy alone (only
    the test of that caching wants it)."""
    old = {key: os.environ.get(key) for key in LEVERS}
    try:
        _set_env(kv, reload=_reload)
        yield
    finally:
        _set_env(old)


@pytest.fixture
def lever():
    """``lever(CCR_2CTA="0", CCR_NO_HIST=None, ...)``: set levers for the rest of the test, effective at once;
    everything is restored and re-read at teardown."""
    stack = contextlib.ExitStack()

    def set_(_reload=True, **kv):
        stack.enter_context(levers(_reload, **kv))

    with stack:
        yield set_


# ---- sortable keys (the kernels' ord32 / ord64 with the top bit flipped: signed order == rank order) ----

def key64(values):
    """int64 keys of float64 ``values`` (torch): larger key == better value, -0.0 just below +0.0."""
    b = values.to(torch.float64).view(torch.int64)
    return torch.where(b < 0, b ^ 0x7FFFFFFFFFFFFFFF, b)


def _key64_np(values):
    b = np.asarray(values, dtype=np.float64).view(np.int64)
    return np.where(b < 0, b ^ np.int64(0x7FFFFFFFFFFFFFFF), b)


def _bits(x, dtype):
    return np.ascontiguousarray(np.asarray(x, dtype=dtype)).view(np.int64 if dtype == np.float64 else np.int32)


# ---- the fused kernel's scores ----

def _pitch_d(t, rows, D):
    """Rows [rows, D] of ``t`` with pitch D: ``t`` itself when it already is that, else a copy (columns
    past D, which the kernels never read, are dropped)."""
    t = t[:rows]
    if t.shape[1] == D and (rows <= 1 or t.stride(0) == D):
        return t
    return t[:, :D].contiguous()


def tc_scores(q, items, D, n_items=None):
    """fp32 [B, N] scores identical to the fused kernel's, from ``ccr_score_dense`` on its tensor-core path.

    ``q`` [B, >= D] and ``items`` [>= N, >= D] are the device-stored rows (``table.encode_queries(Q)`` and
    ``table.data``), bf16 or fp16.  Shapes the dense call would hand to its CUDA-core kernel are made
    tensor-core shapes: the query rows are repeated up to 2^20 scores, zero item rows appended up to 256."""
    from ccr_b200 import engine

    B = q.shape[0]
    N = items.shape[0] if n_items is None else int(n_items)
    out = torch.empty((B, N), dtype=torch.float32, device=q.device)
    if B == 0 or N == 0:
        return out
    qd, it = _pitch_d(q, B, D), _pitch_d(items, N, D)
    if N < ITEM_TILE:
        it = torch.cat([it, torch.zeros((ITEM_TILE - N, D), dtype=it.dtype, device=it.device)])
    n_pad = it.shape[0]
    rows = max(1, min(65535, BLOCK_BYTES // (4 * n_pad)))
    for r0 in range(0, B, rows):
        qb = qd[r0 : r0 + rows]
        nb = qb.shape[0]
        reps = -(-DENSE_TC_MIN // (nb * n_pad))
        if reps > 1:
            assert nb * reps <= 65535, "too few scores for the tensor-core dense path"
            qb = qb.repeat(reps, 1)
        out[r0 : r0 + nb] = engine.score_dense(qb, it, n_items=n_pad, D=D)[:nb, :N]
    return out


def override_values(q, items, indptr, cols, vals, mode, D):
    """float64 [nnz] values the override kernel gives the mask entries, exactly.  q / items: the stored rows
    (torch or numpy, bf16 / fp16 / fp32 holding such values); D: the kernel's D.

    ADD: lane l of one warp sums fmaf over the 8-element chunks c = l, l + 32, ... < D / 8 in order, then an
    xor butterfly with offsets 16 .. 1; a product of two bf16 or two fp16 values is exact in fp32, so each
    fmaf is one rounded fp32 add.  The value is double(lane 0's sum) + the entry's value."""
    indptr = np.asarray(indptr, dtype=np.int64)
    cols = np.asarray(cols, dtype=np.int64)
    vals = np.asarray(vals, dtype=np.float64)
    nnz = int(indptr[-1])
    if mode == MASK_SET:
        return vals[:nnz].copy()
    row_of = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))

    def rows_f32(t, idx):
        if isinstance(t, torch.Tensor):
            return t[torch.as_tensor(idx, device=t.device)][:, :D].float().cpu().numpy()
        return np.asarray(t)[idx][:, :D].astype(np.float32)

    Qe, Ve = rows_f32(q, row_of), rows_f32(items, cols[:nnz])
    n_chunks = D >> 3
    acc = np.zeros((nnz, 32), dtype=np.float32)
    lanes = np.arange(32)
    for t in range(-(-n_chunks // 32)):
        c = lanes + 32 * t
        live = c < n_chunks
        for j in range(8):
            e = c[live] * 8 + j
            acc[:, live] = acc[:, live] + Qe[:, e] * Ve[:, e]
    for off in (16, 8, 4, 2, 1):
        acc = acc + acc[:, lanes ^ off]
    return acc[:, 0].astype(np.float64) + vals[:nnz]


def _mask_host(mask):
    """(indptr, cols, vals, mode) of a SparseMask or such a tuple; None for no mask."""
    if mask is None:
        return None
    if isinstance(mask, tuple):
        return mask
    if mask.mode == MASK_NONE or mask.nnz == 0:
        return None
    ip, c, v = mask.host
    return ip, c, v, mask.mode


def exact_topk(values, k, id_offset=0, allow_short=False, drop_nan=False):
    """Top k of ``values`` [R, N] (torch float32 or float64) under the kernels' order: value descending
    (ord64), then id ascending.  Returns (float64 values, int64 ids + id_offset) [R, k]; with
    ``allow_short`` and k > N the rows end in (-inf, -1).  ``drop_nan``: NaN values never rank (the
    streaming top-k kernels' rule); a row with fewer than k other values ends in (-inf, -1) too."""
    R, N = values.shape
    kk = min(k, N)
    if drop_nan:
        key = key64(values)
        key[torch.isnan(values)] = torch.iinfo(torch.int64).min
        ids = torch.sort(key, dim=1, descending=True, stable=True).indices[:, :kk]
        vals = torch.gather(values, 1, ids).to(torch.float64)
        nan = torch.isnan(vals)
        vals[nan] = -np.inf
        ids = torch.where(nan, torch.full_like(ids, -1 - id_offset), ids)
    elif values.dtype == torch.float32 and N < (1 << 31):
        # one distinct int64 per item: [ord32(score) : ~id], exactly the kernels' 64-bit candidate key
        b = values.view(torch.int32)
        hi = torch.where(b < 0, b ^ 0x7FFFFFFF, b).to(torch.int64)
        key = (hi << 32) | (0xFFFFFFFF - torch.arange(N, device=values.device, dtype=torch.int64))
        top = torch.topk(key, kk, dim=1, sorted=True).values
        ids = 0xFFFFFFFF - (top & 0xFFFFFFFF)
    else:
        ids = torch.sort(key64(values), dim=1, descending=True, stable=True).indices[:, :kk]
    if not drop_nan:
        vals = torch.gather(values, 1, ids).to(torch.float64)
    ids = ids + id_offset
    if kk < k:
        if not allow_short:
            raise ValueError("k > N without allow_short")
        vals = torch.cat([vals, torch.full((R, k - kk), -np.inf, dtype=torch.float64, device=vals.device)], 1)
        ids = torch.cat([ids, torch.full((R, k - kk), -1, dtype=torch.int64, device=ids.device)], 1)
    return vals, ids


def exact_reference(q, items, D, k, mask=None, id_offset=0, allow_short=False, n_items=None, rows=None):
    """(values float64, ids int64) numpy [B, k]: the exact top k the fused tensor-core kernel must return for
    the stored rows ``q`` / ``items`` (device) and ``mask`` (SparseMask or (indptr, cols, vals, mode)).
    ``rows``: only these query rows (sorted int array)."""
    N = items.shape[0] if n_items is None else int(n_items)
    m = _mask_host(mask)
    ovr = None
    if m is not None:
        ip, cols, _, mode = m
        ovr = override_values(q, items, *m, D=D)
        f32 = bool(np.array_equal(ovr.astype(np.float32).astype(np.float64), ovr))
    sel = np.arange(q.shape[0]) if rows is None else np.asarray(rows, dtype=np.int64)
    out_v, out_i = [], []
    block = max(1, BLOCK_BYTES // (4 * max(N, ITEM_TILE)))
    for b0 in range(0, len(sel), block):
        rb = sel[b0 : b0 + block]
        sc = tc_scores(q[torch.as_tensor(rb, device=q.device)], items, D, n_items=N)
        if ovr is not None:
            if not f32:
                sc = sc.double()
            lo, hi = ip[rb], ip[rb + 1]
            n_e = hi - lo
            e = np.repeat(lo - np.concatenate([[0], np.cumsum(n_e)[:-1]]), n_e) + np.arange(int(n_e.sum()))
            r_local = np.repeat(np.arange(len(rb)), n_e)
            dev = sc.device
            sc[torch.as_tensor(r_local, device=dev), torch.as_tensor(cols[e].astype(np.int64), device=dev)] = \
                torch.as_tensor(ovr[e], device=dev).to(sc.dtype)
        v, i = exact_topk(sc, k, id_offset, allow_short)
        out_v.append(v.cpu().numpy())
        out_i.append(i.cpu().numpy())
        del sc
    return np.concatenate(out_v), np.concatenate(out_i)


# ---- checkers: a list of violations, empty when the output is right ----

def check_exact(s, i, d, want_vals, want_ids, limit=5):
    """ids and float64 values equal to the oracle bit for bit (+0.0 is not -0.0), and every float32 score
    the float32 rounding of its value."""
    s = np.asarray(s, dtype=np.float32)
    i = np.asarray(i, dtype=np.int64)
    d = np.asarray(d, dtype=np.float64)
    want_vals = np.asarray(want_vals, dtype=np.float64)
    want_ids = np.asarray(want_ids, dtype=np.int64)
    if i.shape != want_ids.shape or d.shape != want_vals.shape or s.shape != i.shape:
        return [f"shapes: ids {i.shape} values {d.shape} scores {s.shape} vs oracle {want_ids.shape}"]
    errs = []
    bad = (i != want_ids) | (_bits(d, np.float64) != _bits(want_vals, np.float64))
    for r in np.nonzero(bad.any(axis=1))[0][:limit]:
        j = int(np.argmax(bad[r]))
        diff = np.nonzero(bad[r])[0]
        got_only = sorted(set(i[r].tolist()) - set(want_ids[r].tolist()))[:4]
        want_only = sorted(set(want_ids[r].tolist()) - set(i[r].tolist()))[:4]
        errs.append(f"row {r}: {diff.size} ranks differ from rank {j}: got (id {i[r, j]}, {d[r, j]!r}) want "
                    f"(id {want_ids[r, j]}, {want_vals[r, j]!r}); only returned by the kernel {got_only}, "
                    f"only by the oracle {want_only}")
    if int(bad.any(axis=1).sum()) > limit:
        errs.append(f"... {int(bad.any(axis=1).sum())} rows differ in all")
    sb = _bits(s, np.float32) != _bits(d.astype(np.float32), np.float32)
    if sb.any():
        r, j = (int(x[0]) for x in np.nonzero(sb))
        errs.append(f"row {r} rank {j}: float32 score {s[r, j]!r} is not float32({d[r, j]!r})")
    return errs


def check_bounded(s, i, d, q, items, D, k, mask=None, id_offset=0, n_items=None):
    """For the SIMT kernel, whose fp32 summation order is not reproduced: with x_j the float64 sum of the
    stored operands and beta_j = gamma_D * sum|q v| + D * 2^-149 (gamma_D = D u / (1 - D u), u = 2^-24, a
    bound of fp32 round-to-nearest summation in any order), every returned unmasked value is within beta of
    x, mask entries equal the override emulation exactly, ids are unique, the order is strict (value
    descending under ord64, then id ascending), and nothing is missing: every unreturned unmasked item has
    x_j - beta_j <= the k-th value and every unreturned mask entry ranks below the k-th entry."""
    s = np.asarray(s, dtype=np.float32)
    i = np.asarray(i, dtype=np.int64)
    d = np.asarray(d, dtype=np.float64)
    B, kk = i.shape
    N = items.shape[0] if n_items is None else int(n_items)
    errs = []
    if kk != k:
        return [f"{kk} columns returned for k = {k}"]
    qd = q[:B, :D].double()
    it = items[:N, :D].double()
    x = (qd @ it.T).cpu().numpy()
    u = 2.0 ** -24
    gamma = D * u / (1 - D * u) + 2 * D * 2.0 ** -53  # + the float64 reference's own rounding
    beta = (gamma * (qd.abs() @ it.abs().T) + D * 2.0 ** -149).cpu().numpy()
    masked = np.zeros((B, N), dtype=bool)
    ovr_val = {}
    m = _mask_host(mask)
    if m is not None:
        ip, cols, _, _ = m
        ov = override_values(q, items, *m, D=D)
        for r in range(B):
            for e in range(int(ip[r]), int(ip[r + 1])):
                masked[r, cols[e]] = True
                ovr_val[(r, int(cols[e]))] = ov[e]
    sb = _bits(s, np.float32) != _bits(d.astype(np.float32), np.float32)
    if sb.any():
        r, j = (int(v[0]) for v in np.nonzero(sb))
        errs.append(f"row {r} rank {j}: float32 score {s[r, j]!r} is not float32({d[r, j]!r})")
    keys = _key64_np(d)
    for r in range(B):
        if len(errs) >= 5:
            break
        loc = i[r] - id_offset
        if len(set(loc.tolist())) != k or loc.min() < 0 or loc.max() >= N:
            errs.append(f"row {r}: ids not unique or out of range: {i[r][:8].tolist()} ...")
            continue
        order_ok = (keys[r, :-1] > keys[r, 1:]) | ((keys[r, :-1] == keys[r, 1:]) & (loc[:-1] < loc[1:]))
        if not order_ok.all():
            j = int(np.argmin(order_ok))
            errs.append(f"row {r}: ranks {j}, {j + 1} out of order: (id {i[r, j]}, {d[r, j]!r}) then "
                        f"(id {i[r, j + 1]}, {d[r, j + 1]!r})")
        for j, c in enumerate(loc):
            if masked[r, c]:
                if _key64_np(ovr_val[(r, int(c))]) != keys[r, j]:
                    errs.append(f"row {r}: masked id {i[r, j]} has {d[r, j]!r}, override {ovr_val[(r, int(c))]!r}")
            elif abs(d[r, j] - x[r, c]) > beta[r, c]:
                errs.append(f"row {r}: id {i[r, j]} value {d[r, j]!r} is {abs(d[r, j] - x[r, c]):.3e} from its "
                            f"float64 sum, bound {beta[r, c]:.3e}")
        out = np.ones(N, dtype=bool)
        out[loc] = False
        kth, kth_id = d[r, -1], loc[-1]
        miss = np.nonzero(out & ~masked[r] & (x[r] - beta[r] > kth))[0]
        if miss.size:
            c = int(miss[0])
            errs.append(f"row {r}: id {c + id_offset} (float64 sum {x[r, c]!r}, bound {beta[r, c]:.3e}) must "
                        f"outrank the k-th value {kth!r} but was not returned")
        for c in np.nonzero(out & masked[r])[0]:
            v = ovr_val[(r, int(c))]
            if (_key64_np(v), -c) > (_key64_np(kth), -kth_id):
                errs.append(f"row {r}: mask entry {c + id_offset} ({v!r}) outranks the k-th entry but was not "
                            "returned")
                break
    return errs


def check_kernel(algo, s, i, d, q, items, D, k, mask=None, id_offset=0, n_items=None):
    """``check_exact`` against ``exact_reference`` for the tensor-core kernel (algo 2), ``check_bounded`` for
    the CUDA-core kernel (algo 1).  s, i, d: the search's outputs (torch)."""
    s, i, d = (t.cpu().numpy() for t in (s, i, d))
    if algo == 1:
        return check_bounded(s, i, d, q, items, D, k, mask, id_offset=id_offset, n_items=n_items)
    want_v, want_i = exact_reference(q, items, D, k, mask, id_offset=id_offset, n_items=n_items)
    return check_exact(s, i, d, want_v, want_i)


# ---- plan mirrors of the dense and BM25 top-k entries (csrc/ccr_api.cu: dense_plan, bm25_plan) ----
# Neither entry exports its plan; the size queries expose it exactly (ccr_topk_dense_workspace_bytes is the dense
# total, ccr_bm25_topk_workspace_bytes the larger BM25 total), so a test that checks the mirror against them may
# trust its split counts and stream ranges.  Without a device the library plans for 148 SMs.

DEFAULT_SMS = 148
DENSE_SLACK = 4096        # kDenseSlack: columns a dense block scans between two prune checks
FIN_LIST = 4096           # kFinList: finalize's shared-memory entry list
FIN_MAX_STREAMS = 1024    # kFinMaxStreams
BMW_WARPS, BMW_MINI, BMW_BLOCKS_PER_SM, BMW_MAX_TERMS = 8, 512, 4, 32  # warp-private BM25 kernel
BMW_SKETCH_M = 5          # kBmwSketchM
BM_CHUNK, BM_SLACK, BM_BLOCKS_PER_SM = 4096, 1024, 5                   # block-wide BM25 kernel


def cand_capacity(k, slack):
    return (2 * k + slack + 63) // 64 * 64


def carve(*sizes):
    """Total bytes of workspace regions taken one after another, each starting at a 256-byte boundary."""
    off = 0
    for s in sizes:
        off = (off + s + 255) // 256 * 256
    return off


def _ceil(a, b):
    return -(-a // b)


def dense_plan(B, N, k, nnz=0, h=0, sms=DEFAULT_SMS):
    """ccr_topk_dense_f32's plan for k + h candidates per row: S column splits of ``per`` columns each (whole
    4096-column chunks; trailing splits may be empty), C keys per split."""
    rows = max(B, 1)
    S = max(1, min(_ceil(8 * sms, rows), _ceil(N, DENSE_SLACK), FIN_MAX_STREAMS))
    C = cand_capacity(k + h, DENSE_SLACK)
    per = _ceil(_ceil(N, S), DENSE_SLACK) * DENSE_SLACK
    total = carve(rows * S * C * 8, rows * S * 4, nnz * 8, nnz * 4)
    return dict(S=S, C=C, per=per, total=total, k_keep=k + h)


def dense_split_cols(plan, N):
    """[(first column, end)] of every split of a dense plan."""
    return [(min(s * plan["per"], N), min((s + 1) * plan["per"], N)) for s in range(plan["S"])]


def dense_finalize_entries(plan, N, k_row, nnz_row=0):
    """(lo, hi): bounds of the entries finalize gathers for one row with k_row = k + nnz(row) and nnz(row) mask
    records: the splits' candidates, less those in the row's mask (dropped), plus the records.  A split keeps
    every column until its buffer passes C - 4096 keys, then at least k_row and, after a histogram prune of its
    only chunk, at most (k_row + C - 4096) / 2.  When no split prunes, every column is a candidate and each
    masked one is replaced by its record: exactly N."""
    C, lo, hi = plan["C"], 0, 0
    fill = C - DENSE_SLACK
    for a, b in dense_split_cols(plan, N):
        n = b - a
        lo += n if n <= fill else k_row
        if n <= fill:
            hi += n
        elif n <= DENSE_SLACK:
            hi += max(k_row, (k_row + fill) // 2)
        else:
            hi += fill
    if lo == N:
        return N, N
    return lo, hi + nnz_row


def bm25_plan(Bq, N, k, warp, sms=DEFAULT_SMS):
    """ccr_bm25_topk's plan: S doc splits (blocks) per query, ``streams`` candidate lists of C keys per query
    (8 warps per block for the warp-private kernel), ``per`` docs per stream (whole mini-chunks / chunks)."""
    rows = max(Bq, 1)
    if warp:
        s = _ceil(BMW_BLOCKS_PER_SM * sms, rows)
        minis = _ceil(N, BMW_MINI)
        if s * BMW_WARPS > minis:
            s = _ceil(minis, BMW_WARPS)
        s = max(1, min(s, FIN_MAX_STREAMS // BMW_WARPS))
        streams, C = s * BMW_WARPS, cand_capacity(k, BMW_MINI)
        per = _ceil(minis, streams) * BMW_MINI
    else:
        s = max(1, min(_ceil(BM_BLOCKS_PER_SM * sms, rows), _ceil(N, BM_CHUNK), FIN_MAX_STREAMS))
        streams, C = s, cand_capacity(k, BM_SLACK)
        per = _ceil(_ceil(N, BM_CHUNK), s) * BM_CHUNK
    total = carve(rows * streams * C * 8, rows * streams * 4, rows * 4)
    return dict(S=s, streams=streams, C=C, per=per, total=total, warp=warp)


def bm25_stream_docs(plan, N):
    """[(first doc, end)] of every stream of a BM25 plan; the warp-private kernel's block b runs streams
    8b .. 8b + 7."""
    return [(min(s * plan["per"], N), min((s + 1) * plan["per"], N)) for s in range(plan["streams"])]


def bm25_workspace(Bq, N, k, sms=DEFAULT_SMS):
    """ccr_bm25_topk_workspace_bytes: room for either kernel."""
    return max(bm25_plan(Bq, N, k, True, sms)["total"], bm25_plan(Bq, N, k, False, sms)["total"])


# ---- BM25: the float64 accumulation the header specifies ----

def bm25_post_val(tf, idf_t, doc_norm_d, k1):
    """float64 impacts in the header's operation order: ((tf * idf) * (k1 + 1)) * (1 / (tf + doc_norm))."""
    tf = np.asarray(tf, dtype=np.float64)
    return ((tf * idf_t) * (k1 + 1)) * (1.0 / (tf + doc_norm_d))


def bm25_scores(post_indptr, post_docs, post_val, q_indptr, q_terms, N, device="cpu"):
    """float64 [Bq, N] scores: per query a +0.0 accumulator, each term's postings added in q_terms order, one
    add per (term, doc).  Term position j of every query is one scatter: a query has one term there and a term
    one posting per doc, so each cell gets exactly one rounded add per term, in the header's order."""
    dev = torch.device(device)
    ip = torch.as_tensor(np.asarray(post_indptr, dtype=np.int64), device=dev)
    docs = torch.as_tensor(np.asarray(post_docs, dtype=np.int64), device=dev)
    vals = torch.as_tensor(np.asarray(post_val, dtype=np.float64), device=dev)
    q_indptr = np.asarray(q_indptr, dtype=np.int64)
    q_terms = np.asarray(q_terms, dtype=np.int64)
    Bq = len(q_indptr) - 1
    acc = torch.zeros((Bq, N), dtype=torch.float64, device=dev)
    lengths = np.diff(q_indptr)
    for j in range(int(lengths.max()) if Bq else 0):
        qs = np.nonzero(lengths > j)[0]
        terms = torch.as_tensor(q_terms[q_indptr[qs] + j], device=dev)
        lo, n = ip[terms], ip[terms + 1] - ip[terms]
        if int(n.sum()) == 0:
            continue
        q_of = torch.repeat_interleave(torch.as_tensor(qs, device=dev), n)
        first = torch.repeat_interleave(lo - (torch.cumsum(n, 0) - n), n)
        e = first + torch.arange(int(n.sum()), device=dev)
        acc.index_put_((q_of, docs[e]), vals[e], accumulate=True)
    return acc
