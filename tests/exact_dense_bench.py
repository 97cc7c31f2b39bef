"""Rate of the exact dense scores (ccr_score_dense_exact, DESIGN.md section 6b) beside the scan-format dense tiles
(ccr_score_dense_f32 on the bf16 scan copy) and torch's float64 matmul on the same GPU, in one run.

For each (B, N, D): ms per call (CUDA events, after two warm-up calls; mean, min and max over the repetitions)
and GFLOP/s at 2 B N D per call; the exact kernel's rate over torch's FP64 rate.  Prints the card's name and
power limit first, then one JSON line per shape.  Inputs are randn rows generated on the device; the item
tables (0.2-0.8 GB fp32) exceed the 126 MB L2.

    python tests/exact_dense_bench.py [--shapes 1024x262144x768,4096x65536x768] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))

from ccr_b200 import engine  # noqa: E402


def timed(fn, reps):
    """(mean, min, max) ms per call over reps calls after two warm-up calls."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return sum(ms) / len(ms), min(ms), max(ms)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError:
        out = ""
    return out or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1024x262144x768,4096x65536x768")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("exact_dense_bench needs a CUDA device")
    print(json.dumps({"card": card()}), flush=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    for spec in a.shapes.split(","):
        B, N, D = (int(x) for x in spec.split("x"))
        q = torch.randn(B, D, device="cuda", generator=g)
        items = torch.randn(N, D, device="cuda", generator=g)
        q_scan, items_scan = q.bfloat16(), items.bfloat16()
        q64, items64 = q.double(), items.double()
        flop = 2.0 * B * N * D
        res = {"B": B, "N": N, "D": D}
        runs = (("exact", lambda: engine.score_dense_exact(q, items)),
                ("dense_f32_bf16_scan", lambda: engine.score_dense(q_scan, items_scan)),
                ("torch_f64_matmul", lambda: q64 @ items64.T))
        for name, fn in runs:
            mean, lo, hi = timed(fn, a.reps)
            res[name] = {"ms": round(mean, 3), "ms_min": round(lo, 3), "ms_max": round(hi, 3),
                         "gflops": round(flop / mean / 1e6, 1)}
            torch.cuda.empty_cache()
        res["exact_over_torch_f64"] = round(res["exact"]["gflops"] / res["torch_f64_matmul"]["gflops"], 3)
        print(json.dumps(res), flush=True)
        del q, items, q_scan, items_scan, q64, items64
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
