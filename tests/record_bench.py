"""Time of the entry-record kernel that feeds finalize on each of its paths, and of ``engine.topk_dense`` with
an additive prior.

Paths (tables and scores generated on the device, seeded):
  dense  ``engine.topk_dense`` on a materialised fp32 score matrix, 4096 x 262144, k = 100, ADD prior of
         64..256 entries per row (one thread per entry);
  fused  ``EmbeddingTable.search`` on a bf16 table of 1 M x 768, B = 4096, k = 100, ADD prior of 64 entries per
         row (one warp per entry, bf16 dot);
  exact  the same on an exact table with fp16 scan copies (one warp per candidate and mask entry, fp32 rows
         summed in float64).
For each path one JSON line: time per call (CUDA events after one warm-up; mean, min and max over the
repetitions) and, from a separate ``torch.profiler`` run, the device time per call of every kernel whose name
matches --kernels (the record kernel under its current and earlier names).

    python tests/record_bench.py [--paths dense,fused,exact] [--reps 10]
"""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))

import ccr_b200  # noqa: E402
from ccr_b200 import engine  # noqa: E402

KERNELS = r"entry_records_kernel|entry_indptr_kernel|override_kernel|override_dense_kernel|exact_entries_kernel"


def timed(fn, reps):
    """(mean, min, max) ms per call over reps calls after one warm-up."""
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return [round(sum(ts) / len(ts), 3), round(min(ts), 3), round(max(ts), 3)]


def kernel_us(fn, reps, pattern):
    """Device time per call (us) of every kernel whose name matches ``pattern``, over reps profiled calls."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if re.search(pattern, e.key):
            out[e.key] = round(e.device_time_total / reps, 2)
    return out


def prior(B, N, lo, hi, seed):
    """ADD prior: lo..hi random columns per row, values ~ N(0, 0.1)."""
    rs = np.random.RandomState(seed)
    lens = rs.randint(lo, hi + 1, size=B)
    m = engine.SparseMask.from_flat(lens, rs.randint(0, N, size=int(lens.sum())), N, 0.0, engine.MASK_ADD, "cuda")
    vals = torch.as_tensor(rs.standard_normal(m.nnz) * 0.1, device="cuda")
    m.vals.copy_(vals)
    m.host = (m.host[0], m.host[1], vals.cpu().numpy())
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--paths", default="dense,fused,exact")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--kernels", default=KERNELS)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    g = torch.Generator(device="cuda").manual_seed(0)
    B, k, D = 4096, 100, 768
    for path in a.paths.split(","):
        if path == "dense":
            N = 262144
            scores = torch.randn(B, N, device="cuda", generator=g)
            mask = prior(B, N, 64, 256, 1)
            fn = lambda: engine.topk_dense(scores, k, mask=mask)  # noqa: E731
        else:
            N = 1 << 20
            dtype = torch.bfloat16 if path == "fused" else torch.float16
            table = ccr_b200.EmbeddingTable(N, D, device="cuda", dtype=dtype, exact=path == "exact")
            table.append(torch.randn(N, D, device="cuda", generator=g))
            q = table.encode_queries(torch.randn(B, D, device="cuda", generator=g))
            mask = prior(B, N, 64, 64, 1)
            fn = lambda: table.search(q, k, mask=mask, encoded=True)  # noqa: E731
        print(json.dumps({"path": path, "B": B, "N": N, "k": k, "mask_nnz": mask.nnz, "ms": timed(fn, a.reps),
                          "record_kernel_us": kernel_us(fn, a.reps, a.kernels), "reps": a.reps, "gpu": gpu,
                          "lib": os.environ.get("CCR_B200_LIB", "in-tree")}), flush=True)
        del fn, mask
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
