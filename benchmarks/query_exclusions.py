"""Cost of per-query exclusions in the fused top-k (icr_cos_topk_excl), against the same call without them.

C2 (10,000 x 49,688 x 384, k = 100): one fused call per step with 0 / 16 / 256 / 4,096 excluded rows per query, the rows
drawn at random and, separately, each query's own best rows (which moves every bootstrap maximum). The bitmap is built once
(icr_query_exclusion_bits, timed on its own), as a batch job that reuses exclusion sets would. Then request-sized batches on
the same catalog (Q = 8 / 32 / 256, k = 10, 16 rows per query), and 1,000 requests through a recommend() loop against one
recommend_batch() call with a fake encoder. Device times from CUDA events (median of the steps); the card's name and power
limit are read in the same run. Usage: python benchmarks/query_exclusions.py [--steps 20]
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import instacart_next_order_recommendation_b200 as icr  # noqa: E402
from instacart_next_order_recommendation_b200 import ops  # noqa: E402
from oracle import oracle  # noqa: E402

N, D = 49_688, 384


def timed_ms(fn, steps):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in ev)
    return ts[len(ts) // 2]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def own_best(cat, q, n):
    s = torch.nn.functional.normalize(q.float(), dim=1) @ torch.nn.functional.normalize(cat.rows.float(), dim=1).T
    return torch.topk(s, n, dim=1).indices.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--requests", type=int, default=1000)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "c2": {}, "small": {}}
    items = oracle.synth_isotropic(N, D, 1).cuda()
    queries = oracle.synth_isotropic(10_000, D, 2).cuda()
    rng = np.random.default_rng(3)
    for dt in (torch.float32, torch.bfloat16):
        name = "f32" if dt == torch.float32 else "bf16"
        cat = icr.DeviceCatalog(items, dtype=dt)
        q = queries.to(dt)
        kw = dict(cat_planes=cat.planes, cat_inv_norms=cat.inv_norms)
        row = {"none_ms": timed_ms(lambda: ops.cos_topk(q, cat.rows, 100, **kw), args.steps)}
        best = own_best(cat, q, 4096)
        for n in (16, 256, 4096):
            for kind in ("random", "own_best"):
                lists = [rng.choice(N, n, replace=False) for _ in range(q.shape[0])] if kind == "random" else list(best[:, :n])
                bits = ops.query_exclusion_bits(lists, N, cat.device)
                row[f"{kind}_{n}_ms"] = timed_ms(lambda: ops.cos_topk(q, cat.rows, 100, exclude_bits=bits, **kw), args.steps)
                if kind == "random":
                    offs = torch.from_numpy(np.arange(0, (q.shape[0] + 1) * n, n, dtype=np.int64)).cuda()
                    flat = torch.from_numpy(np.concatenate(lists).astype(np.int64)).cuda()
                    row[f"bits_build_{n}_ms"] = timed_ms(lambda: ops.query_exclusion_bits((offs, flat), N, cat.device), args.steps)
        row["random_16_over_none"] = row["random_16_ms"] / row["none_ms"]
        res["c2"][name] = row
        small = {}
        for Q in (8, 32, 256):
            qs = q[:Q].contiguous()
            bits = ops.query_exclusion_bits([rng.choice(N, 16, replace=False) for _ in range(Q)], N, cat.device)
            small[f"Q{Q}_none_us"] = 1e3 * timed_ms(lambda: ops.cos_topk(qs, cat.rows, 10, **kw), 50)
            small[f"Q{Q}_excl16_us"] = 1e3 * timed_ms(lambda: ops.cos_topk(qs, cat.rows, 10, exclude_bits=bits, **kw), 50)
        res["small"][name] = small
        print(json.dumps({name: {"c2": row, "small": small}}), flush=True)

    # recommend() loop against recommend_batch(): the same requests, each with its own 16 excluded products
    table = items.cpu().numpy()

    class FakeEnc:
        def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, convert_to_tensor=False):
            out = table[[int(t[2:]) for t in texts]]
            return torch.from_numpy(out).cuda() if convert_to_tensor else out

    with tempfile.TemporaryDirectory() as tmp:
        corpus = Path(tmp) / "corpus.json"
        pids = [f"p{i}" for i in range(N)]
        corpus.write_text(json.dumps({p: f"c:{i}" for i, p in enumerate(pids)}))
        rec = icr.Recommender("fake-model", corpus, model=FakeEnc(), use_index=False)
        reqs = [f"c:{int(i)}" for i in rng.integers(0, N, args.requests)]
        excl = [set(rng.choice(pids, 16, replace=False).tolist()) for _ in reqs]
        rec.recommend_batch(reqs[:8], exclude_product_ids=excl[:8])
        for r, e in zip(reqs[:8], excl[:8]):
            rec.recommend(r, exclude_product_ids=e)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop = [rec.recommend(r, exclude_product_ids=e) for r, e in zip(reqs, excl)]
        t1 = time.perf_counter()
        batch = rec.recommend_batch(reqs, exclude_product_ids=excl)
        t2 = time.perf_counter()
        res["recommend"] = {"requests": len(reqs), "loop_ms": (t1 - t0) * 1e3, "batch_ms": (t2 - t1) * 1e3, "same_ids": [[p for p, _ in r] for r in loop] == [[p for p, _ in r] for r in batch]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
