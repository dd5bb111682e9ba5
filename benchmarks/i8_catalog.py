"""fp32 vs fp16 vs int8 catalogs: request latency, large-catalog and batch call times, and ranking quality, in one process.

    python benchmarks/i8_catalog.py [out.txt]

Timings alternate the three dtypes round by round (clock and neighbour effects hit all three alike); medians of CUDA-event
times. HBM fraction = the catalog's resident row bytes (N * D * bytes per element) / time / 7.7 TB/s; tensor fraction =
2 * Q * N * D / time / the data-sheet dense rate (int8 4,500 TOPS, fp16 2,250 TFLOP/s, fp32: its one fp16 screening term at
2,250). Both are data-sheet shares, not measured peaks. Recall is the kernels' output against fp64 on the fp32 inputs.
"""
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, ".")
import instacart_next_order_recommendation_b200 as icr  # noqa: E402
from oracle import oracle  # noqa: E402

DTYPES = [("fp32", torch.float32), ("fp16", torch.float16), ("int8", torch.int8)]
ELEM = {"fp32": 4, "fp16": 2, "int8": 1}
PEAK_OPS = {"fp32": 2250e12, "fp16": 2250e12, "int8": 4500e12}
HBM = 7.7e12
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
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e6)
    return float(np.median(ts))


def alternate(fns, reps, rounds, timer):
    res = {n: [] for n in fns}
    for fn in fns.values():
        timer(fn, 3)
    for _ in range(rounds):
        for n, fn in fns.items():
            res[n].append(timer(fn, reps))
    return {n: float(np.median(v)) for n, v in res.items()}


def fractions(n, ms, Q, N, D):
    t = ms * 1e-3
    return N * D * ELEM[n] / t / HBM, 2.0 * Q * N * D / t / PEAK_OPS[n]


def table(title, cases, N, D):
    say(title)
    say()
    say("| case | dtype | ms | HBM fraction | tensor fraction | int8 vs fp16 |")
    say("|---|---|---|---|---|---|")
    for label, Q, r in cases:
        for n, _ in DTYPES:
            h, tfr = fractions(n, r[n], Q, N, D)
            rel = f"{100 * (r['int8'] / r['fp16'] - 1):+.1f} %" if n == "int8" else ""
            say(f"| {label} | {n} | {r[n]:.4f} | {100 * h:.1f} % | {100 * tfr:.1f} % | {rel} |")
    say()


def main():
    torch.cuda.set_device(0)
    say(f"card: {card()}")
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    say()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    # ---- C1: batch-1 requests, cold L2 (catalog copies in rotation), k = 10 -------------------------------------------------
    N, D = 49_688, 384
    items, _ = oracle.synth_clustered(N, D, seed=1234)
    items_d = items.cuda()
    copies = {n: [icr.DeviceCatalog(items_d, dtype=dt) for _ in range(8)] for n, dt in DTYPES}
    q32 = F.normalize(items_d[17:18] + 0.05 * torch.randn(1, D, device="cuda"), dim=1)
    qd = {"fp32": q32, "fp16": q32.half(), "int8": q32}

    def req(n):
        it = iter(range(10**9))
        return lambda: copies[n][next(it) % 8].topk_request(qd[n], 10)

    r = alternate({n: req(n) for n, _ in DTYPES}, 200, 5, host_timed)
    say("## C1 (49,688 x 384): one request, k = 10, 8 catalog copies in rotation (cold L2), host clock around topk_request")
    say()
    say("| dtype | µs | int8 vs fp16 |")
    say("|---|---|---|")
    for n, _ in DTYPES:
        say(f"| {n} | {r[n]:.1f} | {f'{100 * (r[n] / r['fp16'] - 1):+.1f} %' if n == 'int8' else ''} |")
    say()

    # ---- C2: 10,000 x 49,688 x 384, k = 100, L2 flushed ---------------------------------------------------------------------
    q2, _ = oracle.synth_queries_from_items(items, 10_000, seed=99)
    q2 = q2.cuda()
    q2in = {"fp32": q2, "fp16": q2.half(), "int8": q2}
    r = alternate({n: (lambda n=n: copies[n][0].topk(q2in[n], 100)) for n, _ in DTYPES}, 10, 5, lambda fn, reps: timed(fn, reps, flush))
    table("## C2: Q = 10,000, k = 100, L2 flushed, device time", [("C2", 10_000, r)], N, D)
    del copies
    torch.cuda.empty_cache()

    # ---- 10^7 x 768 single-GPU catalog -------------------------------------------------------------------------------------
    NB, DB = 10_000_000, 768
    g = torch.Generator(device="cuda").manual_seed(4)
    big = torch.empty(NB, DB, device="cuda")
    for s0 in range(0, NB, 1_000_000):
        big[s0 : s0 + 1_000_000] = F.normalize(torch.randn(1_000_000, DB, device="cuda", generator=g), dim=1)
    cats = {n: icr.DeviceCatalog(big, dtype=dt) for n, dt in DTYPES}
    cases = []
    for Q in (1, 8, 64, 256):
        qc = F.normalize(big[torch.arange(Q, device="cuda") * 30_011] + 0.3 * torch.randn(Q, DB, device="cuda", generator=g), dim=1)
        qin = {"fp32": qc, "fp16": qc.half(), "int8": qc}
        r = alternate({n: (lambda n=n, qin=qin: cats[n].topk(qin[n], 100)) for n, _ in DTYPES}, 5, 3, lambda fn, reps: timed(fn, reps, flush))
        cases.append((f"Q = {Q}, k = 100", Q, r))
    table(f"## {NB:,} x {DB} catalog (fp16 {NB * DB * 2 / 1e9:.1f} GB, int8 {NB * DB / 1e9:.1f} GB), device time", cases, NB, DB)
    del cats, big
    torch.cuda.empty_cache()

    # ---- recall against fp32 exact -----------------------------------------------------------------------------------------
    say("## Recall against fp64 exact on the fp32 inputs: 256 queries, N = 49,688, D = 384")
    say()
    say("| data | k | fp16 recall | int8 recall |")
    say("|---|---|---|---|")
    for data in ("clustered", "isotropic"):
        if data == "clustered":
            it, _ = oracle.synth_clustered(N, D, seed=1234)
            qs, _ = oracle.synth_queries_from_items(it, 256, seed=1235)
        else:
            it, qs = oracle.synth_isotropic(N, D, seed=1234), oracle.synth_isotropic(256, D, seed=1235)
        ex = F.normalize(qs.double().cuda(), dim=1) @ F.normalize(it.double().cuda(), dim=1).T
        for k in (10, 100):
            ei = torch.topk(ex, k, dim=1).indices.cpu().tolist()
            rec = {}
            for n, dt in DTYPES[1:]:
                _, i = icr.DeviceCatalog(it.cuda(), dtype=dt).topk(qs.cuda() if n == "int8" else qs.cuda().half(), k)
                rec[n] = np.mean([len(set(a) & set(b)) / k for a, b in zip(i.cpu().tolist(), ei)])
            say(f"| {data} | {k} | {rec['fp16']:.4f} | {rec['int8']:.4f} |")
    say()
    say(f"card (again, after the runs): {card()}")
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
