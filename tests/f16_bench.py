#!/usr/bin/env python3
"""Fused-kernel time of fp16 vs bf16 tables on ONE card (manual benchmark; feeds profiles/ and DESIGN.md).

    python tests/f16_bench.py [--batches 1,128,512,4096] [--rounds 3] [--secs 1.0] [--n 8841823] [--out DIR]

Both tables have bench.py's shape (8,841,823 x 768, 13.6 GB each) and rows from bench.py's generator,
one rounded to bf16 and one to fp16, resident in the same process.  Every call is bench.py's step
(top-100, history mask).  For every batch size the two dtypes alternate over ``--rounds`` rounds; in a
round each dtype runs back-to-back calls for ``--secs`` seconds, and the fused score + select kernel of
every call is timed with CUDA events recorded by the library itself (ccr_set_profile_events).  Prints
the card name and power limit, a Markdown table (mean kernel ms per round, both dtypes) and one JSON
line; with ``--out`` writes both there.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))
import torch  # noqa: E402

import bench  # noqa: E402
import ccr_b200  # noqa: E402
from ccr_b200 import _lib, engine  # noqa: E402


def card():
    """Name and power limit of GPU 0 as nvidia-smi reports them (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001 -- the numbers are still worth printing
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})", "max_sm_clock": "unknown"}


def time_window(L, table, q, k, mask, secs):
    """Back-to-back calls for ``secs`` seconds; mean fused-kernel ms."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    table.search(q, k, mask=mask, encoded=True)
    e1.record()
    torch.cuda.synchronize()
    iters = max(5, int(secs * 1e3 / max(e0.elapsed_time(e1), 0.05)))
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in kev:
        L.ccr_set_profile_events(a.cuda_event, b.cuda_event)
        table.search(q, k, mask=mask, encoded=True)
    L.ccr_set_profile_events(None, None)
    torch.cuda.synchronize()
    return statistics.mean(a.elapsed_time(b) for a, b in kev), iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,128,512,4096")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--secs", type=float, default=1.0)
    ap.add_argument("--n", type=int, default=bench.N_ITEMS)
    ap.add_argument("--k", type=int, default=bench.TOPK)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("f16_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}", flush=True)
    tables = {}
    for label, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16)):
        t = ccr_b200.EmbeddingTable(args.n, bench.DIM, device=dev, dtype=dt)
        bench.build_shard(t, 0, args.n, dev)
        tables[label] = t
    torch.cuda.synchronize()
    L = _lib.lib()
    rows = []
    lines = ["| B | bf16 kernel ms (per round) | fp16 kernel ms (per round) | fp16 / bf16 (means) | "
             "bf16 spread | fp16 spread |", "|---|---|---|---|---|---|"]
    for B in (int(b) for b in args.batches.split(",")):
        qf = torch.randn((B, bench.DIM), generator=torch.Generator().manual_seed(7))
        indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, args.n))
        mask = engine.SparseMask(indptr, cols, vals, args.n, engine.MASK_SET, dev)
        qs = {label: t.encode_queries(qf) for label, t in tables.items()}
        for label, t in tables.items():  # warm-up of every shape the windows use
            for _ in range(3):
                t.search(qs[label], args.k, mask=mask, encoded=True)
        torch.cuda.synchronize()
        res = {"bf16": [], "fp16": []}
        for r in range(args.rounds):
            order = ("bf16", "fp16") if r % 2 == 0 else ("fp16", "bf16")
            for label in order:
                ms, iters = time_window(L, tables[label], qs[label], args.k, mask, args.secs)
                res[label].append(ms)
        mb, mf = statistics.mean(res["bf16"]), statistics.mean(res["fp16"])
        sb = (max(res["bf16"]) - min(res["bf16"])) / mb
        sf = (max(res["fp16"]) - min(res["fp16"])) / mf
        rows.append({"B": B, "bf16_ms": res["bf16"], "fp16_ms": res["fp16"], "ratio": mf / mb,
                     "bf16_spread": sb, "fp16_spread": sf})
        line = (f"| {B} | {', '.join(f'{v:.3f}' for v in res['bf16'])} | {', '.join(f'{v:.3f}' for v in res['fp16'])} "
                f"| {mf / mb:.4f} | {sb * 100:.2f} % | {sf * 100:.2f} % |")
        lines.append(line)
        print(line, flush=True)
    head = (f"{info['name']}, power limit {info['power_limit']}; corpus {args.n:,} x {bench.DIM}, k={args.k}, history "
            f"mask; fused score + select kernel (ccr_set_profile_events), mean over >= {args.secs} s of back-to-back "
            f"calls per window, dtypes alternated over {args.rounds} rounds")
    result = {"card": info, "n": args.n, "dim": bench.DIM, "k": args.k, "secs": args.secs, "rounds": args.rounds,
              "rows": rows}
    print(json.dumps(result), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "f16_bench.md"), "w") as f:
            f.write(head + "\n\n" + "\n".join(lines) + "\n")
        with open(os.path.join(args.out, "f16_bench.json"), "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
