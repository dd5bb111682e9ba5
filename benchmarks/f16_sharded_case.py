"""ShardedCatalog(dtype=float16) on N GPUs equals the single-GPU fp16 search (NCCL and peer exchange).

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29523 benchmarks/f16_sharded_case.py
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, ".")
import instacart_next_order_recommendation_b200 as icr  # noqa: E402
from oracle import oracle  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
N, D = 60_013, 384
items, _ = oracle.synth_clustered(N, D, seed=21)
queries, _ = oracle.synth_queries_from_items(items, 64, seed=22)
lo, hi = icr.shard_bounds(N, world, rank)
full = icr.DeviceCatalog(items.to(dev), dtype=torch.float16)
ok = True
for ex in ("nccl", "peer"):
    sh = icr.ShardedCatalog(items[lo:hi], row_offset=lo, total_rows=N, dtype=torch.float16, device=dev, exchange=ex)
    for Q, k in ((1, 10), (7, 100), (64, 100)):
        q = queries[:Q].to(dev)
        v, i = sh.topk(q, k)
        fv, fi = full.topk(q, k)
        torch.cuda.synchronize()
        same = torch.equal(i, fi) and torch.equal(v, fv)
        ok &= same
        if rank == 0:
            print(f"{ex} Q={Q} k={k}: {'equal' if same else 'DIFFERENT'}")
t = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0 and int(t.item()) == 1:
    print("F16_SHARDED_OK")
dist.destroy_process_group()
