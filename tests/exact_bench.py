"""Exact fp32 ranking vs the default scan ranking on the same scan format (DESIGN.md section 6b).

For bf16 and fp16 scans, at the bench workload (8.84 M x 768, B = 4096, k = 100, history mask of 64 items per
row) and the NQ shape (2.68 M x 768, B = 3452, k = 1001), on randn and clustered tables, prints one JSON line
per configuration: time per call (CUDA events, after one warm-up call; mean, min and max over the
repetitions), k', the share of rows certified by the scan stage, the rows that went through the fallback,
and the fallback's own cost: one call with every row sent through it (CCR_EXACT_FALLBACK=1), per row.
Tables are generated on the device.

    python tests/exact_bench.py [--shapes bench,nq] [--tables randn,clustered] [--scans fp16,bf16] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))

import ccr_b200  # noqa: E402
from ccr_b200 import _lib, engine  # noqa: E402

SHAPES = {"bench": (8841823, 4096, 100, 64), "nq": (2681468, 3452, 1001, 0)}
D = 768


def gen(kind, n, g, centers):
    if kind == "randn":
        return torch.randn(n, D, device="cuda", generator=g)
    idx = torch.randint(0, centers.shape[0], (n,), device="cuda", generator=g)
    return centers[idx] + 0.5 * torch.randn(n, D, device="cuda", generator=g)


def timed(fn, reps):
    """(mean, min, max) ms per call over reps calls after one warm-up, and the last output."""
    fn()
    torch.cuda.synchronize()
    ts, out = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return (sum(ts) / len(ts), min(ts), max(ts)), out


def fallback_ms_per_row(table, q32, k, mask, rows=256):
    """One exact call with every row through the fallback, on the first ``rows`` query rows."""
    os.environ["CCR_EXACT_FALLBACK"] = "1"
    _lib.reload_env()
    try:
        m = mask.rows(0, rows) if mask is not None else None
        (ms, _, _), _ = timed(lambda: table._search_exact(q32[:rows], k, mask=m, encoded=True), 1)
    finally:
        os.environ.pop("CCR_EXACT_FALLBACK")
        _lib.reload_env()
    return ms / rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="bench,nq")
    ap.add_argument("--tables", default="randn,clustered")
    ap.add_argument("--scans", default="fp16,bf16")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    for shape in a.shapes.split(","):
        N, B, k, h = SHAPES[shape]
        for kind in a.tables.split(","):
            g = torch.Generator(device="cuda").manual_seed(0)
            centers = torch.randn(1000, D, device="cuda", generator=g) * 1.0
            for scan in a.scans.split(","):
                dtype = torch.float16 if scan == "fp16" else torch.bfloat16
                table = ccr_b200.EmbeddingTable(N, D, device="cuda", dtype=dtype, exact=True)
                for s in range(0, N, 1 << 20):
                    table.append(gen(kind, min(N, s + (1 << 20)) - s, g, centers))
                q32 = table.encode_queries(gen(kind, B, g, centers))
                q_scan = torch.empty(q32.shape, dtype=dtype, device="cuda")
                table._scan_copy(q32, q_scan)
                mask = None
                if h:
                    rows = torch.randint(0, N, (B, h), generator=torch.Generator().manual_seed(1)).numpy()
                    mask = engine.SparseMask.from_lists(rows, N, -1e6, engine.MASK_SET, "cuda")
                t_plain, _ = timed(lambda: engine.score_topk(q_scan, table.data, k, mask=mask, n_items=table.n,
                                                             D=table.ld), a.reps)
                t_exact, out = timed(lambda: table._search_exact(q32, k, mask=mask, encoded=True), a.reps)
                fb_row = fallback_ms_per_row(table, q32, k, mask)
                n_fb = out[-1]
                print(json.dumps({
                    "shape": shape, "table": kind, "scan": scan, "N": N, "B": B, "k": k, "mask_per_row": h,
                    "k_cand": _lib.exact_k_candidates(B, N, table.ld, k, _lib.FLAG_F16 if scan == "fp16" else 0),
                    "ms_default": [round(t, 2) for t in t_plain], "ms_exact": [round(t, 2) for t in t_exact],
                    "certified_share": round(1 - n_fb / B, 4), "fallback_rows": n_fb,
                    "fallback_ms_per_row": round(fb_row, 3), "reps": a.reps, "gpu": gpu}), flush=True)
                del table, q32, q_scan
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
