#!/usr/bin/env python3
"""A/B of several builds of libccr_b200 on bench.py's resident step, in one process and one CUDA context.

    python tests/ring_depth_ab.py --libs old=/path/a.so,new=/path/b.so [--rounds 5] [--steps 20] [--warmup 3]
                                  [--shapes 4096:100,1024:100] [--out DIR]

Every build is loaded from its own path (the way CCR_B200_LIB selects one) and runs bench.py's step on bench.py's
inputs: the same seeded corpus (8,841,823 x 768 bf16), queries and history mask (set -1e6).  The builds are timed
in alternating order, `--rounds` times each, so that drift of the clock under the power cap spreads over all of
them.  Per cell: ms per step (CUDA events around `--steps` back-to-back steps), the fused kernel's ms (the
library's profiling events), the median NVML SM clock sampled during the timed steps; once per run: the card's
name and power limit.  The last step's [B, k] scores and ids of every build are compared bit for bit with the
first build's.  Writes DIR/ring_depth_ab.md (table) and DIR/ring_depth_ab.json (every sample).

Every build is loaded through this tree's ccr_b200._lib binding, so every build must export the symbols that
binding declares and report its ABI version.  profiles/r03_ring_depth_ab.md was taken with it.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))

import torch  # noqa: E402

import bench  # noqa: E402


def card_info(index):
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        name = pynvml.nvmlDeviceGetName(h)
        name = name.decode() if isinstance(name, bytes) else name
        return {"name": name, "power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0,
                "sm_max_mhz": pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)}
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "nvml": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", required=True, help="name=path,... (the first build is the reference of the output check)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="4096:100", help="B:k,... on bench.py's corpus and mask")
    ap.add_argument("--out", default="ring_depth_ab_out")
    a = ap.parse_args()
    libs = [tuple(s.split("=", 1)) for s in a.libs.split(",") if s]
    shapes = [tuple(int(x) for x in s.split(":")) for s in a.shapes.split(",") if s]

    import ccr_b200
    from ccr_b200 import _lib, engine

    if not torch.cuda.is_available():
        raise RuntimeError("ring_depth_ab.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    def use_lib(path):
        _lib.LIB_PATH = path
        _lib._lib = None
        return _lib.lib()

    use_lib(libs[0][1])  # builds the inputs
    N, D = bench.N_ITEMS, bench.DIM
    index = ccr_b200.ShardedIndex(N, D, device=dev)
    table = index.table
    bench.build_shard(table, index.lo, index.hi, dev)
    b_max = max(b for b, _ in shapes)
    q_all = table.encode_queries(torch.randn((b_max, D), generator=torch.Generator().manual_seed(7)))
    masks = {}
    for b, _ in shapes:
        if b not in masks:
            indptr, cols, vals = bench.rows_to_csr(bench.history_mask_rows(b, N))
            masks[b] = engine.SparseMask(indptr, cols, vals, N, engine.MASK_SET, dev)
    info = card_info(0)

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    for e in [x for p in kev for x in p]:
        e.record()
    samples, ref_out, check = [], {}, {}
    for r in range(a.rounds):
        order = libs if r % 2 == 0 else libs[::-1]
        for name, path in order:
            L = use_lib(path)
            for b, k in shapes:
                q, mask = q_all[:b], masks[b]  # a smaller B takes the first B of the same seeded queries
                plan = _lib.plan_info(b, N, D, k, mask_nnz=mask.nnz, mask_max_row_nnz=mask.max_row_nnz)
                for _ in range(a.warmup):
                    table.search(q, k, mask=mask, encoded=True)
                torch.cuda.synchronize()
                with bench.ClockSampler(0) as clk:
                    ev0.record()
                    for it in range(a.steps):
                        L.ccr_set_profile_events(kev[it][0].cuda_event, kev[it][1].cuda_event)
                        out = table.search(q, k, mask=mask, encoded=True)
                    L.ccr_set_profile_events(None, None)
                    ev1.record()
                    torch.cuda.synchronize()
                ms = ev0.elapsed_time(ev1) / a.steps
                kern = statistics.mean(x.elapsed_time(y) for x, y in kev)
                s, i = out[0].cpu(), out[1].cpu()
                if r == 0 and name == libs[0][0]:  # round 0 runs the first build first
                    ref_out[(b, k)] = (s, i)
                rs, ri = ref_out[(b, k)]
                bad = int((s.view(torch.int32) != rs.view(torch.int32)).sum()) + int((i != ri).sum())
                c = check.setdefault(f"{name}:B{b}:k{k}", {"vs": libs[0][0], "differing_elements": 0, "cells": 0})
                c["differing_elements"] += bad
                c["cells"] += 1
                clocks = clk.summary()
                row = {"round": r, "lib": name, "B": b, "k": k, "ms_per_step": ms, "kernel_ms": kern,
                       "queries_per_s": b / ms * 1e3, "sm_mhz": clocks.get("sm_mhz"),
                       "throttle": clocks.get("reasons"), "plan": plan, "differing_elements": bad}
                samples.append(row)
                print(json.dumps(row), flush=True)

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "ring_depth_ab.json"), "w") as f:
        json.dump({"card": info, "libs": dict(libs), "steps": a.steps, "warmup": a.warmup, "samples": samples,
                   "output_check": check}, f, indent=1)
    lines = [f"card: {info.get('name')}, power limit {info.get('power_limit_w')} W, max SM clock "
             f"{info.get('sm_max_mhz')} MHz; corpus {N:,} x {D} bf16, history mask (set -1e6), bench.py's seeds; "
             f"{a.rounds} alternating rounds x {a.steps} steps per cell",
             "",
             "| B | k | build | ms/step median (min-max) | kernel ms median | queries/s median (min-max) | SM MHz median | "
             "outputs vs first build |",
             "|---|---|---|---|---|---|---|---|"]
    for b, k in shapes:
        for name, _ in libs:
            rows = [x for x in samples if x["lib"] == name and x["B"] == b and x["k"] == k]
            ms = [x["ms_per_step"] for x in rows]
            qps = [x["queries_per_s"] for x in rows]
            km = [x["kernel_ms"] for x in rows]
            mhz = [x["sm_mhz"] for x in rows if x["sm_mhz"]]
            c = check[f"{name}:B{b}:k{k}"]
            lines.append(f"| {b} | {k} | {name} | {statistics.median(ms):.3f} ({min(ms):.3f}-{max(ms):.3f}) | "
                         f"{statistics.median(km):.3f} | {statistics.median(qps):,.0f} ({min(qps):,.0f}-{max(qps):,.0f}) | "
                         f"{statistics.median(mhz) if mhz else 'n/a'} | "
                         f"{'identical' if c['differing_elements'] == 0 else str(c['differing_elements']) + ' differ'} |")
    text = "\n".join(lines) + "\n"
    with open(os.path.join(a.out, "ring_depth_ab.md"), "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
