#!/usr/bin/env python3
"""Batch sweep x variant A/B on ONE box (builder tool; feeds profiles/r02_*.md).

    python tests/perf_sweep.py --batches 256,512,4096 --variants "base=;single=CCR_2CTA=0" [--k 100] [--mask 1]
                               [--n 8841823] [--secs 0.4] [--md out.md]

The table is built once (bench.py's generator).  For every batch size the variants are run round-robin
(`--rounds` rounds of back-to-back calls, each round `--secs` long) so that clock / thermal drift hits
them equally.  Per (B, variant): ms per call (CUDA events around the whole public call: seeding
pre-pass, fused kernel, overrides, finalize), ms of the fused kernel alone (ccr_set_profile_events),
median SM clock while it ran, queries/s and the fraction of the binding roofline
min(tensor peak, HBM bandwidth over the corpus bytes) at the MEASURED_PEAKS burst figures.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import ccr_b200  # noqa: E402
from ccr_b200 import _lib, engine  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="256,512,1024,4096")
ap.add_argument("--variants", default="base=")
ap.add_argument("--k", type=int, default=100)
ap.add_argument("--mask", type=int, default=0)
ap.add_argument("--n", type=int, default=bench.N_ITEMS)
ap.add_argument("--secs", type=float, default=0.4)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--md", default=None)
args = ap.parse_args()

pk = bench.peaks()
F, BW = pk["tflops_burst"] * 1e12, pk["hbm"] * 1e9
dev = torch.device("cuda:0")
table = ccr_b200.EmbeddingTable(args.n, bench.DIM, device=dev)
bench.build_shard(table, 0, args.n, dev)
variants = []
for spec in args.variants.split(";"):
    name, _, envs = spec.partition("=")
    variants.append((name, dict(e.split("=", 1) for e in envs.split(",") if e)))
ALL_KEYS = {k_ for _, env in variants for k_ in env}

import pynvml  # noqa: E402

pynvml.nvmlInit()
nv = pynvml.nvmlDeviceGetHandleByIndex(0)
samples, stop = [], threading.Event()


def sampler():
    while not stop.is_set():
        samples.append((time.time(), pynvml.nvmlDeviceGetClockInfo(nv, pynvml.NVML_CLOCK_SM)))
        time.sleep(0.005)


threading.Thread(target=sampler, daemon=True).start()
L = _lib.lib()
lines = ["| B | variant | ms/call | kernel ms | SM MHz | queries/s | bound | frac of roofline | kernel frac |",
         "|---|---|---|---|---|---|---|---|---|"]
print("\n".join(lines), flush=True)
for B in (int(b) for b in args.batches.split(",")):
    q = table.encode_queries(torch.randn((B, bench.DIM), generator=torch.Generator().manual_seed(7)))
    mask = None
    if args.mask:
        indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(B, args.n))
        mask = engine.SparseMask(indptr, cols, vals, args.n, engine.MASK_SET, dev)
    t_min = max(2.0 * B * args.n * bench.DIM / F, args.n * bench.DIM * 2 / BW)
    bound = "tensor" if 2.0 * B * bench.DIM / F > bench.DIM * 2 / BW else "hbm"
    res = {name: [] for name, _ in variants}
    for rnd in range(args.rounds):
        for name, env in variants:
            for k_ in ALL_KEYS:
                os.environ.pop(k_, None)
            os.environ.update(env)
            _lib.reload_env()
            for _ in range(2):
                table.search(q, args.k, mask=mask, encoded=True)
            torch.cuda.synchronize()
            # how many calls fit the time slice
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            table.search(q, args.k, mask=mask, encoded=True)
            e1.record()
            torch.cuda.synchronize()
            iters = max(3, min(200, int(args.secs * 1e3 / max(e0.elapsed_time(e1), 0.05))))
            kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
            for a, b in kev:
                a.record(), b.record()
            torch.cuda.synchronize()
            t0 = time.time()
            e0.record()
            for a, b in kev:
                L.ccr_set_profile_events(a.cuda_event, b.cuda_event)
                table.search(q, args.k, mask=mask, encoded=True)
            L.ccr_set_profile_events(None, None)
            e1.record()
            torch.cuda.synchronize()
            t1 = time.time()
            clk = [c for (t, c) in samples if t0 <= t <= t1]
            res[name].append((e0.elapsed_time(e1) / iters, statistics.mean(a.elapsed_time(b) for a, b in kev),
                              statistics.median(clk) if clk else float("nan")))
    for name, _ in variants:
        ms = min(r[0] for r in res[name])
        kms = min(r[1] for r in res[name])
        mhz = statistics.median(r[2] for r in res[name])
        line = (f"| {B} | {name} | {ms:.3f} | {kms:.3f} | {mhz:.0f} | {B / ms * 1e3:,.0f} | {bound} | "
                f"{t_min * 1e3 / ms:.3f} | {t_min * 1e3 / kms:.3f} |")
        lines.append(line)
        print(line, flush=True)
stop.set()
for k_ in ALL_KEYS:
    os.environ.pop(k_, None)
if args.md:
    with open(args.md, "w") as f:
        f.write(f"corpus {args.n:,} x {bench.DIM} bf16, k={args.k}, mask={'history' if args.mask else 'none'}; peaks: "
                f"{pk['tflops_burst']} TFLOP/s burst, {pk['hbm']} GB/s ({pk['source']}); best of {args.rounds} rounds of "
                f"{args.secs} s back-to-back calls per cell\n\n" + "\n".join(lines) + "\n")
