"""fp32 vs bf16 vs fp16 catalogs: request latency, batch throughput and ranking quality, measured in one process.

    python benchmarks/f16_catalog.py [out.txt]

Every timing alternates the three dtypes (a round of fp32, bf16, fp16, repeated) so that clock and neighbour effects hit all
three alike; medians of CUDA-event times. The accuracy table is the kernels' output against fp64 arithmetic on the fp32
inputs (SURVEY §8d generators, seed 1234).
"""
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, ".")
import instacart_next_order_recommendation_b200 as icr  # noqa: E402
from instacart_next_order_recommendation_b200 import ops  # noqa: E402
from oracle import oracle  # noqa: E402

DTYPES = [("fp32", torch.float32), ("bf16", torch.bfloat16), ("fp16", torch.float16)]
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def timed(fn, reps, flush=None):
    """median ms of fn() over reps, CUDA events around each call (flush: zeroed before each call, outside the window)."""
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def host_timed(fn, reps):
    """median us of a call that ends in a host synchronisation (the request paths return host lists)."""
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e6)
    return float(np.median(ts))


def alternate(make_fn, reps, rounds, timer):
    """{dtype: median} with the dtypes interleaved round by round."""
    res = {n: [] for n, _ in DTYPES}
    fns = {n: make_fn(n, dt) for n, dt in DTYPES}
    for fn in fns.values():  # warm-up: graphs, prepared calls, attributes
        timer(fn, 3)
    for _ in range(rounds):
        for n, _ in DTYPES:
            res[n].append(timer(fns[n], reps))
    return {n: float(np.median(v)) for n, v in res.items()}


def row(label, r, unit):
    say(f"| {label} | " + " | ".join(f"{r[n]:.1f}" if unit == "us" else f"{r[n]:.3f}" for n, _ in DTYPES)
        + f" | {100 * (r['fp16'] / r['bf16'] - 1):+.1f} % |")


def main():
    torch.cuda.set_device(0)
    say(f"card: {card()}")
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    say()
    N, D = 49_688, 384
    items, _ = oracle.synth_clustered(N, D, seed=1234)
    items_d = items.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    # ---- C1 requests, cold: rotating over catalog copies that together exceed the 126 MB L2 ------------------------------
    copies = {n: [icr.DeviceCatalog(items_d, dtype=dt) for _ in range(8)] for n, dt in DTYPES}
    q32 = F.normalize(items_d[17:18] + 0.05 * torch.randn(1, D, device="cuda"), dim=1)
    qn = {n: (q32 if dt == torch.float32 else (ops.normalized_f16(q32) if dt == torch.float16 else q32.to(dt))) for n, dt in DTYPES}
    say("## C1 (49,688 x 384), one request, k = 10, 8 catalog copies in rotation (cold L2), host clock around the request")
    say()
    say("| path | fp32 µs | bf16 µs | fp16 µs | fp16 vs bf16 |")
    say("|---|---|---|---|---|")
    for label, use32 in (("topk_request, query in the catalog's dtype", False), ("Recommender path: topk_request, fp32 query", True)):
        def make(n, dt, use32=use32):
            it = iter(range(10**9))
            cats = copies[n]
            q = q32 if use32 else qn[n]
            return lambda: cats[next(it) % 8].topk_request(q, 10)
        row(label, alternate(make, 200, 5, host_timed), "us")
    say()

    # ---- C1 batches ---------------------------------------------------------------------------------------------------------
    say("## C1 batches (device time, CUDA events, L2 warm)")
    say()
    say("| shape | fp32 ms | bf16 ms | fp16 ms | fp16 vs bf16 |")
    say("|---|---|---|---|---|")
    for Q, k in ((32, 10), (64, 100)):
        qb, _ = oracle.synth_queries_from_items(items, Q, seed=Q)
        qb = qb.cuda()
        def make(n, dt, qb=qb, k=k):
            cat, q = copies[n][0], ops._like_catalog(qb, dt)
            return lambda: cat.topk(q, k)
        row(f"Q = {Q}, k = {k}", alternate(make, 50, 5, timed), "ms")
    # ---- C2: 10,000 queries, k = 100, L2 flushed ----------------------------------------------------------------------------
    q2, _ = oracle.synth_queries_from_items(items, 10_000, seed=99)
    q2 = q2.cuda()
    def make_c2(n, dt):
        cat, q = copies[n][0], ops._like_catalog(q2, dt)
        return lambda: cat.topk(q, 100)
    r = alternate(make_c2, 20, 5, lambda fn, reps: timed(fn, reps, flush))
    row("C2: Q = 10,000, k = 100, L2 flushed", r, "ms")
    del copies
    torch.cuda.empty_cache()
    say()

    # ---- C4-shaped shard: 1.25M x 768 ---------------------------------------------------------------------------------------
    say("## C4 shard (1,250,000 x 768, streams from HBM), k = 100, device time")
    say()
    say("| Q | fp32 ms | bf16 ms | fp16 ms | fp16 vs bf16 |")
    say("|---|---|---|---|---|")
    g = torch.Generator(device="cuda").manual_seed(4)
    big = F.normalize(torch.randn(1_250_000, 768, device="cuda", generator=g), dim=1)
    cats = {n: icr.DeviceCatalog(big, dtype=dt) for n, dt in DTYPES}
    for Q in (1, 64, 256):
        qc = F.normalize(big[torch.arange(Q, device="cuda") * 4001] + 0.3 * torch.randn(Q, 768, device="cuda", generator=g), dim=1)
        def make(n, dt, qc=qc):
            cat, q = cats[n], ops._like_catalog(qc, dt)
            return lambda: cat.topk(q, 100)
        row(f"{Q}", alternate(make, 20, 5, lambda fn, reps: timed(fn, reps, flush)), "ms")
    del cats, big
    torch.cuda.empty_cache()
    say()

    # ---- accuracy of the kernels' output -------------------------------------------------------------------------------------
    say("## Ranking quality of the kernels' output: 1,000 queries against fp64 on the fp32 inputs (N = 49,688, D = 384, seed 1234)")
    say()
    say("| data, k | bf16: id set = exact | fp16: id set = exact | bf16 max abs score err | fp16 max abs score err |")
    say("|---|---|---|---|---|")
    for data in ("clustered", "isotropic"):
        if data == "clustered":
            it, _ = oracle.synth_clustered(N, D, seed=1234)
        else:
            it = oracle.synth_isotropic(N, D, seed=1234)
        qs, _ = oracle.synth_queries_from_items(it, 1000, seed=1235) if data == "clustered" else (oracle.synth_isotropic(1000, D, seed=1235), None)
        ex = F.normalize(qs.double().cuda(), dim=1) @ F.normalize(it.double().cuda(), dim=1).T
        for k in (10, 100):
            ev, ei = torch.topk(ex, k, dim=1)
            cells = {}
            for n, dt in DTYPES[1:]:
                cat = icr.DeviceCatalog(it.cuda(), dtype=dt)
                v, i = cat.topk(qs.cuda(), k)
                same = np.mean([set(a) == set(b) for a, b in zip(i.cpu().tolist(), ei.cpu().tolist())])
                err = float((v.double() - ex.gather(1, i)).abs().max())
                cells[n] = (same, err)
            say(f"| {data}, k = {k} | {100 * cells['bf16'][0]:.1f} % | {100 * cells['fp16'][0]:.1f} % | {cells['bf16'][1]:.1e} | {cells['fp16'][1]:.1e} |")
    say()
    say(f"card (again, after the runs): {card()}")
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
