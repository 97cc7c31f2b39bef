#!/usr/bin/env python3
"""Multi-GPU check of exact tables (run under torchrun on a GPU box; tests/test_gpu_exact.py spawns it):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 tests/dist_exact_check.py
A row-sharded ShardedIndex(exact=True) must return what ONE exact table returns, bit for bit (fp32 scores,
ids and float64 values), on every rank, with and without a SET block mask, for host and device queries."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "crowd-coachable-recommendations_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import ccr_b200  # noqa: E402

local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device(f"cuda:{local}")
dist.init_process_group("nccl", device_id=dev)
rank, world = dist.get_rank(), dist.get_world_size()
ok = True
CASES = [
    # N, D, B, k, SET mask?, queries on the host?
    (200_003, 768, 300, 100, False, True),
    (200_003, 768, 300, 100, True, False),
    (1_200_000, 128, 700, 100, True, True),   # seeded + histogram + CTA pairs per shard
    (1_500, 768, 9, 1001, True, True),
    (7, 64, 5, 7, False, True),               # fewer rows than ranks: empty shards, k == N
]
for (N, D, B, k, masked, host_q) in CASES:
    g = torch.Generator().manual_seed(N + D)
    P = torch.randn((N, D), generator=g)
    Q = torch.randn((B, D), generator=g)
    rs = np.random.RandomState(N)
    mask = None
    if masked:
        rows = [np.unique(rs.randint(0, N, size=rs.randint(0, min(N, 50)))) for _ in range(B)]
        mask = ccr_b200.SparseMask.from_lists(rows, N, -1e6, ccr_b200.MASK_SET, dev)
    full = ccr_b200.EmbeddingTable.from_tensor(P, device=dev, dtype=torch.float16, exact=True)
    s1, i1, d1 = full.search(Q, k, mask=mask, want_f64=True)
    idx = ccr_b200.ShardedIndex(N, D, device=dev, dtype=torch.float16, exact=True)
    idx.add_local(P[idx.lo:idx.hi])
    assert idx.table.exact
    s2, i2, d2 = idx.search(Q if host_q else Q.to(dev), k, mask=mask)
    same = bool(torch.equal(i1, i2)) and bool(torch.equal(s1, s2)) and bool(torch.equal(d1, d2))
    print(f"rank {rank}/{world} N={N} D={D} B={B} k={k} masked={masked} shard=[{idx.lo},{idx.hi}) "
          f"exact_equal_single_table={same}", flush=True)
    ok &= same
flag = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if int(flag.item()) == 1 else 1)
