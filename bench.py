#!/usr/bin/env python3
"""Benchmark of the score-and-rank hot path (see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config marco|c5] [--batch B]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of B synthetic queries: fused
score(Q . P^T) -> history mask (set -1e6) -> per-row top-k.

--config marco (default; BASELINE.json configs[2], the configuration the metric is quoted on; fits one
    B200): 8,841,823 x 768 bf16 corpus, top-100.  With N > 1 the corpus is row-sharded (strong scaling:
    the corpus is fixed).
--config c5 (BASELINE.json configs[4]): 100,000,000 x 768 bf16 row-sharded over the ranks (19.2 GB each at
    8 GPUs; needs >= 8 GPUs of 180 GB -- or 1 GPU for a single 12.5 M-row shard with --n-items), top-1000.

With N > 1 every rank computes its local top-k as packed 8-byte (float32 score, uint32 global id) keys; an
all-to-all hands every rank the runs of its B/G query rows, an on-device G-way merge-path merge and an
all-gather of the merged rows complete the result on every rank.

value  : queries/s, whole job, inputs (bf16 table shard, bf16 queries, mask CSR) resident in HBM.
e2e    : the same through the public host API from HOST buffers: pinned fp32 queries (each rank uploads
         and encodes 1/G of the rows, all-gathered over NVLink) + the mask CSR are copied H2D, the mask
         is column-sharded on the device, and rank 0 copies the [B,k] scores + ids back D2H, all inside
         the timed region.

--dump-outputs DIR writes the [B,k] scores (float32) and global ids (float64) of the last timed resident
step as DIR/scores.npy and DIR/ids.npy (above 60 MB, a fixed seeded sample of rows, numbered in
DIR/rows.npy).  Every input is generated from fixed seeds, so two builds run with the same arguments can be
compared output for output.  Inside the tree, bench_out/ is the directory git ignores for this.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_ITEMS, DIM, TOPK = 8_841_823, 768, 100
CHUNK = 1 << 20
CONFIGS = {
    "marco": dict(n_items=N_ITEMS, k=100, batch=4096,
                  metric="queries/s, top-100 over 8.8M x 768 corpus",
                  workload="MS-MARCO-shape retrieval (BASELINE.json configs[2]): 8,841,823 x 768 bf16 corpus, "
                           "top-100 with history mask (set -1e6, nnz/row ~ min(Geom(1/8),64))"),
    "c5": dict(n_items=100_000_000, k=1000, batch=4096,
               metric="queries/s, top-1000 over 100M x 768 corpus row-sharded across the GPUs",
               workload="BASELINE.json configs[4]: synthetic 100,000,000 x 768 bf16 item table row-sharded across "
                        "the ranks, top-1000 with history mask, packed all-gather + on-device merge"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="marco", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="queries per step (default: the config's)")
    ap.add_argument("--n-items", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's scores / ids as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    cfg = CONFIGS[a.config]
    a.custom_shape = a.n_items is not None or a.k is not None
    a.batch = a.batch or cfg["batch"]
    a.n_items = a.n_items or cfg["n_items"]
    a.k = a.k or cfg["k"]
    a.metric = cfg["metric"] if not a.custom_shape else f"queries/s, top-{a.k} over {a.n_items} x {DIM} corpus"
    a.workload = cfg["workload"] if not a.custom_shape else (
        f"custom shape: {a.n_items} x {DIM} bf16 corpus, top-{a.k} with history mask")
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=p.get("bf16_tflops_sustained", 1401.9), tflops_burst=p.get("bf16_tflops", 1667.8),
                    hbm=p.get("hbm_gbs", 6445.3), source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def measured_traffic(key):
    """DRAM bytes per launch of the dominant kernel on a named workload, from the committed ncu capture
    (profiles/traffic.json: {key: {"dram_bytes": read + write, "source": file}}); None when no capture of
    this exact workload exists."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, None
    ent = json.load(open(path)).get(key)
    return (ent["dram_bytes"], ent["source"]) if ent else (None, None)


def history_mask_rows(B, n_items, seed=2):
    """SURVEY.md §8d C3: per-row nnz ~ min(Geometric(1/8), 64), columns uniform."""
    rs = np.random.RandomState(seed)
    return [np.unique(rs.randint(0, n_items, size=min(64, rs.geometric(1.0 / 8)))) for _ in range(B)]


def rows_to_csr(rows):
    indptr = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in rows], out=indptr[1:])
    cols = np.concatenate(rows).astype(np.int32) if len(rows) else np.zeros(0, np.int32)
    return indptr, cols, np.full(len(cols), -1e6)


DUMP_BYTES = 60 * 10**6  # under 64 MB with room for the .npy headers


def dump_outputs(out_dir, arrays, limit=DUMP_BYTES):
    """Write host arrays (float32 / float64, one row per query) as out_dir/<name>.npy.  When they hold more
    than `limit` bytes, the same fixed, seeded sample of rows is taken from each and the sampled row
    numbers are written as rows.npy."""
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{name}: {a.dtype} (float32 / float64 only)")
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > limit:
        keep = limit // (row_bytes + 8)
        rows = np.sort(np.random.RandomState(0).choice(n, size=keep, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


# ----------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own CPU path (oracle port)
# ----------------------------------------------------------------------------------------------
def host_corpus(n_items, seed=0):
    """fp32 host corpus of the workload's shape for the CPU legs.  One seeded 1 Mi-row normal block is
    drawn and repeated with a per-copy scale (distinct rows, normal-like scores): drawing 6.8 G normals
    with the serial CPU generator would take longer than the measurement."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn((min(n_items, CHUNK), DIM), generator=g)
    if n_items <= CHUNK:
        return base
    P = torch.empty((n_items, DIM))
    for c, s in enumerate(range(0, n_items, CHUNK)):
        e = min(n_items, s + CHUNK)
        torch.mul(base[: e - s], 1.0 + 1e-3 * c, out=P[s:e])
    return P


def cpu_reference_step(P, n_queries, seed=0):
    from oracle import ccr_oracle as O

    g = torch.Generator().manual_seed(100 + seed)
    Q = torch.randn((n_queries, DIM), generator=g)
    rows = history_mask_rows(n_queries, P.shape[0], seed=2)
    t0 = time.perf_counter()
    O.ranking_core_ref(Q, P, batch_size=512, block_rows=rows, sim_type="dot")
    return time.perf_counter() - t0


REF_WHAT = ("oracle.ranking_core_ref (ms_marco_eval.py:203-230 on CPU: fp32 tile matmul batch 512 -> host QxN matrix "
            "-> -1e6 block mask -> full per-row sort -> top 1001)")


def cpu_baseline(n_items, sample_items=1 << 20, sample_queries=96):
    """Bounded sample for the `ours` line (10-30 s of CPU work): full embedding width, a 1 Mi-row slice of
    the corpus, scaled linearly in the corpus length (`--impl reference` runs the real length)."""
    dt = cpu_reference_step(host_corpus(sample_items), sample_queries)
    qps_sample = sample_queries / dt
    return {
        "value": qps_sample * sample_items / n_items,
        "unit": "queries/s",
        "cores": torch.get_num_threads(),
        "kind": "port",
        "sample": (f"{REF_WHAT} on {sample_queries} queries x {sample_items} items x {DIM}: {dt:.2f} s = "
                   f"{qps_sample:.2f} q/s, scaled linearly by {sample_items}/{n_items} to the full corpus; "
                   f"os.cpu_count()={os.cpu_count()}, affinity={len(os.sched_getaffinity(0))}"),
    }


def workload_config(args, world, shard_rows):
    """`config` of the JSON line: names the workload only, identical for both arms (the product's launch
    plan is a separate top-level key)."""
    return {"workload": args.workload, "n_items": args.n_items, "dim": DIM, "k": args.k,
            "queries_per_step": args.batch, "parallelism": f"row-shard x{world}",
            "l2": f"inputs larger than L2 ({shard_rows * DIM * 2 / 1e9:.1f} GB table shard streamed every step)"}


def reference_sample_queries(n_steps, n_items, budget_s=200.0):
    """Queries per reference step such that `n_steps` steps end within a few minutes on ~16 host cores:
    measured there, a step costs ~2.8 s (17 k tile matmuls over the 27 GB table, independent of the number of
    queries) + ~0.7 s per query (full sort of N scores), both proportional to the corpus length.  The fixed
    part is amortised over fewer queries than the reference's own runs (thousands), so a small sample
    under-states the reference by up to ~25 % (32 queries per step: 1.27 q/s; 8: ~0.95 q/s)."""
    scale = n_items / N_ITEMS
    q = int((budget_s / max(1, n_steps) - 2.8 * scale) / (0.7 * scale))
    return max(1, min(32, q))


def run_reference(args):
    """The reference's CPU implementation of the path at the workload's REAL corpus length (host fp32 table:
    27.2 GB for 8,841,823 x 768): exactly --warmup + --steps steps, each a bounded sample of the workload's
    query batch (sized so the whole run ends within a few minutes); falls back to a corpus sample only if the
    host cannot hold the table."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    n_ref, scale, note = args.n_items, 1.0, "full corpus length"
    try:
        if args.n_items * DIM * 4 > 64 << 30:
            raise MemoryError("corpus above 64 GB of host fp32")
        P = host_corpus(args.n_items)
    except (MemoryError, RuntimeError) as e:  # host too small: bounded corpus sample, scaled linearly
        n_ref = 1 << 20
        scale = n_ref / args.n_items
        note = f"host could not hold the corpus ({type(e).__name__}): {n_ref}-row sample scaled linearly"
        P = host_corpus(n_ref)
    steps, warm = max(1, args.steps), max(0, args.warmup)
    n_queries = reference_sample_queries(steps + warm, n_ref)
    for i in range(warm):
        cpu_reference_step(P, n_queries, seed=1000 + i)
    t0 = time.perf_counter()
    for i in range(steps):
        cpu_reference_step(P, n_queries, seed=i)
    dt = (time.perf_counter() - t0) / steps
    qps = n_queries / dt * scale
    sample = (f"{REF_WHAT}: every step = {n_queries} of the workload's {args.batch} queries x {n_ref} items "
              f"({note}); os.cpu_count()={os.cpu_count()}, affinity={len(os.sched_getaffinity(0))}")
    line = {
        "impl": "reference", "metric": args.metric, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, -(-args.n_items // world)),
        "sample_queries_per_step": n_queries,
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.stop = [], threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:  # noqa: BLE001
            self.nv = None
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv:
            self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()

    def summary(self):
        if not self.nv or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        nv = self.nv
        clk = sorted(s[0] for s in self.samples)
        bits = 0
        for s in self.samples:
            bits |= s[1]
        names = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks": 0x2}
        return {"sm_mhz": clk[len(clk) // 2], "sm_max_mhz": nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM),
                "reasons": [n for n, b in names.items() if bits & b]}


def build_shard(table, lo, hi, dev):
    """Rows [lo, hi) of the synthetic corpus, generated on the device chunk by chunk with a seed per
    global chunk so that any sharding yields the same global table (never materialised on the host)."""
    import ccr_b200  # noqa: F401

    c0, c1 = lo // CHUNK, (hi + CHUNK - 1) // CHUNK
    for c in range(c0, c1):
        g = torch.Generator(device=dev).manual_seed(1000 + c)
        rows = torch.randn((CHUNK, DIM), generator=g, device=dev)
        a, b = max(lo, c * CHUNK), min(hi, (c + 1) * CHUNK)
        table.append(rows[a - c * CHUNK : b - c * CHUNK])
        del rows


def library_baseline(table, q_dev, k, steps=2, chunk=1 << 17):
    """The library-call GPU implementation of the same step on the same box (context, BASELINE.md §3): stock
    torch bf16 ``Q @ P_chunk.T`` (cuBLAS) + ``torch.topk`` per chunk + a final merge.  No mask (it would
    only add work); ranks bf16-rounded scores.  Timed with CUDA events after one warm-up step."""
    items, n = table.data, len(table)

    def step():
        best_s, best_i = [], []
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            v, i = (q_dev @ items[s:e].T).topk(min(k, e - s), dim=1)
            best_s.append(v)
            best_i.append(i + s)
        v, i = torch.cat(best_s, 1), torch.cat(best_i, 1)
        top, pos = v.topk(k, dim=1)
        return top, torch.gather(i, 1, pos)

    step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": q_dev.shape[0] / ms * 1e3, "unit": "queries/s", "ms_per_step": ms, "steps": steps,
            "what": f"torch bf16 Q@P_chunk.T (cuBLAS) + torch.topk per {chunk}-row chunk + merge, no mask, this GPU's "
                    "shard only"}


def run_ours(args):
    import torch.distributed as dist

    import ccr_b200
    from ccr_b200 import _lib, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, N, k = args.batch, args.n_items, args.k
    pk = peaks()
    shard_rows = -(-N // world)
    if shard_rows * DIM * 2 > 170e9:
        raise RuntimeError(f"--config {args.config}: a shard of {shard_rows} rows ({shard_rows * DIM * 2 / 1e9:.1f} GB) "
                           f"does not fit one B200; run it on more GPUs (c5 is defined on 8)")

    # ---- resident state: table shard, queries, mask ----
    index = ccr_b200.ShardedIndex(N, DIM, device=dev)     # world == 1: one shard holding everything
    table, lo, hi = index.table, index.lo, index.hi
    build_shard(table, lo, hi, dev)
    gq = torch.Generator().manual_seed(7)
    q_host = torch.randn((B, DIM), generator=gq).pin_memory()
    rows = history_mask_rows(B, N)
    indptr, cols, vals = rows_to_csr(rows)
    mask_global = engine.SparseMask(indptr, cols, vals, N, engine.MASK_SET, dev)
    mask_local = mask_global.column_shard_device(lo, hi) if world > 1 else mask_global
    q_dev = table.encode_queries(q_host)
    pin = {n: torch.as_tensor(a).pin_memory() for n, a in (("indptr", indptr), ("cols", cols), ("vals", vals))}
    out_s_host = torch.empty((B, k), dtype=torch.float32).pin_memory()
    out_i_host = torch.empty((B, k), dtype=torch.int64).pin_memory()

    def step_resident():
        if world > 1:
            return index._exchange_keys(index._local_topk_keys(q_dev, k, mask_local), k)
        return table.search(q_dev, k, mask=mask_local, encoded=True)

    def step_e2e():
        m = engine.SparseMask.from_device_tensors(pin["indptr"].to(dev, non_blocking=True),
                                                  pin["cols"].to(dev, non_blocking=True),
                                                  pin["vals"].to(dev, non_blocking=True), (indptr, cols, vals), N,
                                                  engine.MASK_SET, f32_exact=True)
        if world > 1:
            s, i, _ = index.search(q_host, k, mask=m)   # host queries: 1/G uploaded per rank + all-gather
        else:
            s, i = table.search(q_host.to(dev, non_blocking=True), k, mask=m)
        if rank == 0:
            out_s_host.copy_(s, non_blocking=True)
            out_i_host.copy_(i, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-only timing through the profiling hook ----
    ev_k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev_k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for e in ev_k0 + ev_k1:
        e.record()  # materialise the cudaEvent_t handles
    L = _lib.lib()

    for _ in range(args.warmup):
        step_resident()
    barrier()
    with ClockSampler(local) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for it in range(args.steps):
            L.ccr_set_profile_events(ev_k0[it].cuda_event, ev_k1[it].cuda_event)
            out = step_resident()
        L.ccr_set_profile_events(None, None)
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(ev_k0, ev_k1)]))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"scores": out[0].cpu().numpy(),
                                         "ids": out[1].cpu().numpy().astype(np.float64)})

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        step_e2e()  # ends with a stream synchronize: rank 0's host has the step's [B,k] result
    g1.record()
    barrier()
    e2e_ms_total = g0.elapsed_time(g1)

    if world > 1:
        t = torch.tensor([ms_total, e2e_ms_total, kern_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_ms_total, kern_ms = t.tolist()
    ms_step = ms_total / args.steps
    value = B / ms_step * 1e3
    e2e_value = B / (e2e_ms_total / args.steps) * 1e3

    n_local = hi - lo
    clocks = clk.summary()
    flops = 2.0 * B * n_local * DIM            # algorithmic flops of one launch of the dominant kernel
    hbm_bytes = float(n_local) * DIM * 2        # algorithmic bytes: the shard once
    t_tensor, t_hbm = flops / (pk["tflops_burst"] * 1e12), hbm_bytes / (pk["hbm"] * 1e9)
    plan = _lib.plan_info(B, n_local, DIM, k, mask_nnz=int(indptr[-1]), mask_max_row_nnz=mask_global.max_row_nnz)
    launches_per_step = plan["n_kernel_launches"] + (2 if world > 1 else 0)   # + merge + key unpack; NCCL kernels not counted
    # which cuBLAS peak the kernel is compared with: the sustained (power-capped) figure when the sampled
    # clock shows the cap at work, the burst figure when the GPU ran un-capped
    capped = "sw_power_cap" in clocks.get("reasons", []) or (clocks.get("sm_mhz") or 0) < 1600
    if t_tensor >= t_hbm:
        achieved = flops / (kern_ms * 1e-3) / 1e12
        peak = pk["tflops"] if capped else pk["tflops_burst"]
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_source": pk["source"] + (", sustained cuBLAS bf16 (sw_power_cap active / clock below 1.6 GHz)"
                                               if capped else ", burst cuBLAS bf16 (clock un-capped)"),
                "frac_of_burst_peak": achieved / pk["tflops_burst"], "algorithmic_flops_per_launch": flops}
    else:
        achieved = hbm_bytes / (kern_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"],
                "peak_source": pk["source"] + ", device copy bandwidth", "algorithmic_bytes_per_launch": hbm_bytes}
    traffic, traffic_src = measured_traffic(f"{args.config}:B{B}:N{n_local}:k{k}:g{world}")
    roof.update({"traffic": traffic, "traffic_source": traffic_src,
                 "kernel": "select_tc_kernel (TMA + tcgen05 GEMM fused with mask + exact top-k)", "kernel_ms": kern_ms})
    line = {
        "metric": args.metric, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, world, shard_rows), "plan": plan,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "queries/s",
                # per rank: its 1/G slice of the fp32 queries + the mask CSR; back: rank 0's [B,k] scores + ids
                "h2d_bytes_per_step": int(-(-B // world) * DIM * 4 + indptr.nbytes + cols.nbytes + vals.nbytes),
                "d2h_bytes_per_step": int(B * k * 12)},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof,
        "step_roofline_frac_of_burst": max(t_tensor, t_hbm) * 1e3 / ms_step,
    }
    if rank == 0 and world == 1 and not args.no_library_baseline:
        line["gpu_library_baseline"] = library_baseline(table, q_dev, k)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(N)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
