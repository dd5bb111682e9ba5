#!/usr/bin/env python
"""Headline benchmark: top-k queries/sec of the retrieval hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload at every N: BASELINE.json configs[1] — batched IR evaluation, 10,000 queries against the
49,688 x 384 fp32 catalog, top-100 (one "step" = one pass over one 10,000-query batch). With N > 1 every
rank holds a replica of the catalog and its own query batch (queries are independent units: weak scaling,
NO data-path collective — the headline `value` says nothing about a collective).

The path that does have an exchange step is measured at EVERY N, including 1, as the `sharded` object: the
FIXED-TOTAL catalogs of BASELINE configs 4 and 5 (10M x 768 bf16 with Q = 1 / 64 / 1024, 100M x 384 bf16 with
Q = 4096), row-sharded over the N GPUs (strong scaling), local fused top-k -> candidate exchange (NVLink
peer-memory kernel, NCCL all-gather timed beside it) -> device merge, with a torch fp32 witness on sampled
queries. `c1` = the batch-1 request of config 1 (cold and graph-replay latency against the HBM roofline),
`c3` = the MNRL step of config 3 (fwd+bwd, B = 256) next to PyTorch eager on the same GPU.

Prints ONE JSON line (rank 0). `value` = device-resident throughput; `e2e` = through the public API with
pinned-host queries in and host results out, copies inside the timed region; `roofline` = the dominant
kernel against the measured bf16 tensor peak (or HBM peak for the GEMV path); `cpu_baseline` = the oracle
port of the reference path (sentence-transformers cos_sim + torch.topk) on this box's host cores.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

C2 = dict(Q=10_000, N=49_688, D=384, k=100)
CATALOG_SEED, QUERY_SEED = 1234, 4321
METRIC = "top-k queries/sec (IR-eval batch: 10,000 queries x 49,688x384 fp32 catalog, top-100)"


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock and throttle reasons sampled every ~5 ms (NVML) while the timed regions run."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index: int):
        self.index, self.sm, self.max_mhz, self.reasons, self.stop, self.thread = index, [], None, set(), False, None

    def __enter__(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def run():
                while not self.stop:
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        bits = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        self.reasons.update(n for b, n in self.REASONS.items() if bits & b)
                    except Exception:
                        pass
                    time.sleep(0.005)

            self.thread = threading.Thread(target=run, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.thread:
            self.thread.join(timeout=2)

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def _cpu_reference_qps(sample_queries: int, budget_s: float, threads: int | None = None):
    """The reference's CPU path for this workload (oracle port): cos_sim -> torch.topk(100), all host threads."""
    import torch

    from oracle import oracle

    if threads:
        torch.set_num_threads(threads)
    items = oracle.synth_isotropic(C2["N"], C2["D"], CATALOG_SEED)
    queries = oracle.synth_isotropic(sample_queries, C2["D"], QUERY_SEED)
    oracle.cos_topk(queries[:64], items, C2["k"])  # warm the thread pool
    done, t0 = 0, time.perf_counter()
    while done < sample_queries:
        oracle.cos_topk(queries[done : done + 500], items, C2["k"], sorted=False)
        done += min(500, sample_queries - done)
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    # best case for the CPU (SURVEY §8d): operands converted and normalised once, outside the timed region
    cn = torch.nn.functional.normalize(items, dim=1).t().contiguous()
    qn = torch.nn.functional.normalize(queries, dim=1)
    done2, t1 = 0, time.perf_counter()
    while done2 < sample_queries and time.perf_counter() - t1 < budget_s / 2:
        torch.topk(torch.mm(qn[done2 : done2 + 500], cn), C2["k"], dim=1, largest=True, sorted=False)
        done2 += min(500, sample_queries - done2)
    best = done2 / (time.perf_counter() - t1)
    return done / dt, done, torch.get_num_threads(), best


def run_reference(args, rank: int):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; sentence-transformers is
    not installable here), rank 0 only, each step a bounded sample of the C2 batch."""
    if rank != 0:
        return
    import torch

    from oracle import oracle

    # all the host threads the process may use: torchrun exports OMP_NUM_THREADS=1 to its workers, which would time a
    # single-threaded CPU baseline whenever the driver launches this arm with N > 1
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, OSError):
        torch.set_num_threads(max(1, os.cpu_count() or 1))
    sample = 500
    items = oracle.synth_isotropic(C2["N"], C2["D"], CATALOG_SEED)
    queries = oracle.synth_isotropic(sample, C2["D"], QUERY_SEED)
    for _ in range(args.warmup):
        oracle.cos_topk(queries, items, C2["k"], sorted=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle.cos_topk(queries, items, C2["k"], sorted=False)
    dt = time.perf_counter() - t0
    qps = sample * args.steps / dt
    cores = torch.get_num_threads()
    sample_desc = f"{sample} of the 10,000 queries per step against the full 49,688x384 fp32 catalog; cos_sim (normalize both + mm) + torch.topk(100, sorted=False), torch CPU"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: 10,000 queries x 49,688x384 fp32 catalog, top-100 (bounded sample per step)", "Q": C2["Q"], "N": C2["N"], "D": C2["D"], "k": C2["k"]},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample_desc, "host_cpus": os.cpu_count()},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline, e2e and kernel-timing loops; the sharded, c1, c3 and ir_eval objects keep their own fixed counts")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"], help="catalog storage dtype (headline: f32, the reference's)")
    ap.add_argument("--path", default="auto", choices=["auto", "gemv", "gemm"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the row-sharded strong-scaling object (configs 4 and 5)")
    ap.add_argument("--no-side", action="store_true", help="skip the c1 / c3 / ir_eval side objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's result of the last timed step of the headline path (DeviceCatalog.topk on the seeded C2 inputs) "
                         "as DIR/topk_values.npy (float32 [Q, k]) and DIR/topk_ids.npy (float64 [Q, k]), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # stdout carries exactly ONE line, the JSON record: native libraries write there too (NCCL prints its version banner
    # on the first collective), so file descriptor 1 is pointed at stderr for the run and the record goes to the saved one
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    import instacart_next_order_recommendation_b200 as icr
    from instacart_next_order_recommendation_b200 import ops

    assert torch.cuda.is_available(), "bench.py needs a B200"
    if world > 1 and os.environ.get("ICR_BENCH_BIND", "1") != "0":
        # pin this rank (and the pinned host buffers it allocates next) to the CPUs NVML reports as local to its GPU:
        # with 8 ranks the end-to-end leg moves ~22 GB/s per rank across PCIe, and remote-socket staging costs bandwidth
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
        except Exception:
            pass
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    path = {"auto": ops.PATH_AUTO, "gemv": ops.PATH_GEMV, "gemm": ops.PATH_GEMM}[args.path]
    tdtype = torch.float32 if args.dtype == "f32" else torch.bfloat16
    Q, N, D, k = C2["Q"], C2["N"], C2["D"], C2["k"]

    # ---- synthetic inputs (isotropic unit vectors, SURVEY §8d(i)); catalog replica per rank, distinct queries per rank
    g = torch.Generator(device=dev).manual_seed(CATALOG_SEED)
    items = torch.nn.functional.normalize(torch.randn(N, D, device=dev, generator=g), dim=1)
    g.manual_seed(QUERY_SEED + rank)
    queries = torch.nn.functional.normalize(torch.randn(Q, D, device=dev, generator=g), dim=1)
    catalog = icr.DeviceCatalog(items, dtype=tdtype)
    queries_dev = queries.to(tdtype)
    queries_host = queries.cpu().pin_memory()
    out_v_host = torch.empty(Q, k, dtype=torch.float32).pin_memory()
    out_i_host = torch.empty(Q, k, dtype=torch.int64).pin_memory()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_device():
        return catalog.topk(queries_dev, k, path=path)

    def step_e2e():
        # public host-to-host API: pinned queries -> H2D -> fused top-k -> D2H of (scores, ids), pieces pipelined on 2 streams
        catalog.topk_host(queries_host, k, out=(out_v_host, out_i_host), path=path)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        barrier()
        for s in range(steps):
            flush.zero_()  # evict L2 between timed iterations (not timed)
            out = None  # the previous step's result is freed before the next one allocates, as when no result is kept
            starts[s].record()
            out = fn()
            stops[s].record()
        barrier()
        ms = [a.elapsed_time(b) for a, b in zip(starts, stops)]
        total = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return total.item(), ms, out

    def timed_in_flight(steps, depth=3):
        """Host-to-host batches kept in flight: the upload of batch s+1 overlaps the kernels of batch s and the download of batch
        s-1 (DeviceCatalog.topk_host(join=False)). ONE timed region around all `steps` batches; every batch's H2D and D2H copies
        and an L2 flush in front of its kernels (on the stream the kernels run on) are inside it."""
        outs = [(torch.empty(Q, k, dtype=torch.float32).pin_memory(), torch.empty(Q, k, dtype=torch.int64).pin_memory()) for _ in range(depth)]
        catalog.topk_host(queries_host, k, out=outs[0], path=path)  # creates the side streams
        rank_stream = catalog._side_streams[1]
        flush_e2e = flush[: 256 << 20]  # 2x the 126 MB L2; this flush is INSIDE the timed region (0.07 ms per batch)
        cur = torch.cuda.current_stream(dev)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        done = []
        barrier()
        t0.record()
        rank_stream.wait_event(t0)
        for s in range(steps):
            if s >= depth:
                done[s - depth].synchronize()  # the consumer has this batch's results; its buffers are free again
            with torch.cuda.stream(rank_stream):
                flush_e2e.zero_()
            done.append(catalog.topk_host(queries_host, k, out=outs[s % depth], path=path, join=False, n_chunks=1)[2])
        cur.wait_event(done[-1])
        t1.record()
        barrier()
        total = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return total.item()

    for _ in range(args.warmup):
        step_device()
    launches_per_step = ops.last_launch_count()
    with ClockSampler(local_rank) as clocks:  # spans every timed region below
        total_ms, per_step, last_out = timed(step_device, args.steps)
        for _ in range(3):
            step_e2e()
        e2e_sync_ms, _, _ = timed(step_e2e, args.steps)
        timed_in_flight(min(args.steps, 4))
        e2e_ms = timed_in_flight(args.steps)
        # ---- dominant kernel alone (CUDA events recorded by the library around that kernel's launches) ---------
        kt = ops.kernel_timing(step_device, args.steps, flush=flush)
    if args.dump_outputs and rank == 0:
        import numpy as np

        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        values, ids = last_out
        np.save(out_dir / "topk_values.npy", values.float().cpu().numpy())
        np.save(out_dir / "topk_ids.npy", ids.double().cpu().numpy())  # float64 holds every row id exactly
    peaks = _peaks()
    flops = 2.0 * Q * N * D
    if kt["kernel"] == "gemm_topk":
        roof = {"bound": "tensor", "achieved": flops / (kt["ms_per_step"] * 1e-3) / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s"}
        roof["note"] = f"algorithmic 2*Q*N*D flops; fp32 parity costs {kt.get('mma_terms', 1)} fp16 MMA terms per flop; peak = {peaks['source']} bf16 burst"
    else:
        # GEMV passes re-read the catalog once per group of <=7 queries: bytes are per launch
        bytes_per_launch = N * D * (4 if args.dtype == "f32" else 2)
        roof = {"bound": "hbm", "achieved": bytes_per_launch / (kt["ms_per_launch"] * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
        roof["note"] = f"catalog bytes per GEMV launch (L2-resident after the first pass); peak = {peaks['source']} HBM copy"
    roof["frac"] = roof["achieved"] / roof["peak"]
    if roof["bound"] == "tensor" and peaks.get("bf16_tflops_sustained"):  # SURVEY 8(d): report against the burst figure and state the sustained one
        roof["peak_sustained"] = peaks["bf16_tflops_sustained"]
        roof["frac_of_sustained"] = roof["achieved"] / peaks["bf16_tflops_sustained"]
    roof["whole_step_frac"] = (flops / (total_ms / args.steps * 1e-3) / 1e12 / peaks["bf16_tflops"]) if roof["bound"] == "tensor" else None
    roof["traffic"] = None  # NOT measured by this run: bytes per launch from the committed ncu --set full capture of this workload, if there is one
    try:
        cap = json.loads((ROOT / "profiles" / "r02_kernel_traffic.json").read_text())[kt["kernel"]][args.dtype]
        if args.path == "auto":
            roof["traffic"] = sum(cap["launch_bytes"]) / len(cap["launch_bytes"])
            roof["traffic_source"] = "static: " + cap.get("source", "ncu --set full capture committed under profiles/") + " (mean dram read+write bytes per launch; not re-measured in this run)"
    except (OSError, KeyError, ValueError, TypeError):
        pass
    roof["kernel"] = kt["kernel"]
    roof["kernel_ms_per_step"] = kt["ms_per_step"]
    roof["kernel_launches_per_step"] = kt["launches_per_step"]

    ir_eval = None
    if world == 1 and not args.no_side:
        try:
            ir_eval = bench_ir_eval(icr, ops, dev, rank, flush)
        except Exception as e:  # a side measurement must not cost the headline line
            ir_eval = {"error": f"{type(e).__name__}: {e}"[:300]}

    c1 = c3 = None
    if world == 1 and not args.no_side:
        for name, fn in (("c1", bench_c1), ("c3", bench_c3)):
            try:
                res = fn(icr, ops, dev, flush)
            except Exception as e:  # a side measurement must not cost the headline line
                res = {"error": f"{type(e).__name__}: {e}"[:300]}
            if name == "c1":
                c1 = res
            else:
                c3 = res
    del catalog, items, queries, queries_dev
    torch.cuda.empty_cache()

    sharded = None
    if not args.no_sharded:
        try:
            sharded = bench_sharded(icr, ops, dist, dev, rank, world, flush)
        except Exception as e:
            if world > 1:
                raise  # ranks must not diverge around collectives
            sharded = {"error": f"{type(e).__name__}: {e}"[:300]}

    value = world * Q * args.steps / (total_ms * 1e-3)
    e2e_in_flight = world * Q * args.steps / (e2e_ms * 1e-3)
    e2e_one = world * Q * args.steps / (e2e_sync_ms * 1e-3)
    e2e = max(e2e_in_flight, e2e_one)  # both go through DeviceCatalog.topk_host with every copy timed; eight ranks on one host gain nothing from batches in flight
    line = {
        "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": "C2: batched IR eval, 10,000 queries x 49,688x384 catalog, top-100 (BASELINE.json configs[1])",
                   "Q_per_gpu": Q, "N": N, "D": D, "k": k, "catalog_dtype": args.dtype, "path": args.path,
                   "multi_gpu": ("catalog replica + own query batch per rank: NO data-path collective in `value` - the collective path is the `sharded` object"
                                 if world > 1 else "single GPU"),
                   "l2": "512 MiB buffer zeroed between timed iterations (L2 flush)", "seeds": [CATALOG_SEED, QUERY_SEED]},
        "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": Q * D * 4, "d2h_bytes_per_step": Q * k * 12,
                "form": "batches_in_flight" if e2e_in_flight >= e2e_one else "one_batch_at_a_time",
                "batches_in_flight": e2e_in_flight, "one_batch_at_a_time": e2e_one,
                "note": "DeviceCatalog.topk_host: pinned-host fp32 queries in, (scores f32, ids i64) out to pinned host through upload / rank / download "
                        "streams; catalog resident in HBM as the reference keeps its index in "
                        "memory. value = the better of the two forms below (`form` says which). batches_in_flight: up to 3 whole batches in flight (join=False, one piece per batch: the upload of batch s+1 and the download of "
                        "batch s-1 run under the kernels of batch s), ONE timed region around all steps, each batch's copies and a 256 MiB L2 flush (2x L2) "
                        "in front of its kernels inside it; one_batch_at_a_time: every batch waits for the one before and is cut into 3 pieces (15/70/15 %) "
                        "that pipeline inside it (per-batch events, flush outside them) - the round-1/2 number"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof,
        "clocks": clocks.summary(),
        "ms_per_step_min": min(per_step),
    }
    if sharded is not None:
        line["sharded"] = sharded
    if c1 is not None:
        line["c1"] = c1
    if c3 is not None:
        line["c3"] = c3
    if ir_eval is not None:
        line["ir_eval"] = ir_eval
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        qps, nq, cores, best = _cpu_reference_qps(sample_queries=4000, budget_s=15.0)
        line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "host_cpus": os.cpu_count(),
                                "sample": f"{nq} of the 10,000 queries against the full catalog: oracle port of cos_sim + torch.topk(100), torch CPU "
                                          "(as called: both operands re-normalised per 500-query call)",
                                "best_case_value": best, "best_case": "operands pre-normalised once, mm + topk only"}
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    if rank == 0:
        os.write(real_stdout, (json.dumps(line) + "\n").encode())


def bench_ir_eval(icr, ops, dev, rank, flush):
    """BASELINE config 2 as the evaluator runs it: embeddings resident -> fused top-100 -> metric kernel -> the metric
    means on the host (recall@10 / NDCG@10 / MRR@10 / MAP@100 from planted relevance on the clustered generator)."""
    import numpy as np
    import torch

    Q, N, D, k = C2["Q"], C2["N"], C2["D"], C2["k"]
    g = torch.Generator(device=dev).manual_seed(CATALOG_SEED + 7)
    centres = torch.nn.functional.normalize(torch.randn(134, D, device=dev, generator=g), dim=1) * (D ** 0.5) * 0.25
    assign = torch.randint(0, 134, (N,), device=dev, generator=g)
    items = torch.nn.functional.normalize(centres[assign] + torch.randn(N, D, device=dev, generator=g), dim=1)
    src = torch.randint(0, N, (Q,), device=dev, generator=g)
    queries = torch.nn.functional.normalize(items[src] + 0.05 * 4.0 / D ** 0.5 * torch.randn(Q, D, device=dev, generator=g), dim=1)
    # relevant(q) = the item q was generated from + up to 4 items of the same cluster
    order = torch.argsort(assign).cpu().numpy()
    a_np, src_np = assign.cpu().numpy(), src.cpu().numpy()
    starts = np.searchsorted(a_np[order], np.arange(135))
    rng = np.random.default_rng(QUERY_SEED)
    rel = []
    for q in range(Q):
        c = a_np[src_np[q]]
        mates = order[starts[c] : starts[c + 1]]
        rel.append(np.concatenate([[src_np[q]], rng.choice(mates, size=min(4, len(mates)), replace=False)]))
    table = ops.RelevanceTable(rel, device=dev)
    catalog = icr.DeviceCatalog(items)
    specs = [(ops.METRIC_RECALL, 10), (ops.METRIC_NDCG, 10), (ops.METRIC_MRR, 10), (ops.METRIC_MAP, 100)]

    def step():
        _, ids = catalog.topk(queries, k)
        means, _ = ops.ir_metrics(ids, table, specs)
        return means.tolist()  # device -> host read of the 4 means; synchronises

    for _ in range(3):
        vals = step()
    ts = []
    for _ in range(10):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        vals = step()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return {"workload": "C2 as the evaluator runs it: 10,000 query and 49,688 corpus embeddings in HBM -> top-100 -> recall/NDCG/MRR/MAP on the device "
                        "-> 4 floats to the host (wall clock incl. the read-back)",
            "ms_per_eval": ts[len(ts) // 2], "queries_per_s": Q / (ts[len(ts) // 2] * 1e-3),
            "recall@10": vals[0], "ndcg@10": vals[1], "mrr@10": vals[2], "map@100": vals[3]}


def bench_c1(icr, ops, dev, flush):
    """BASELINE config 1: one query against the 49,688 x 384 fp32 catalog, top-10 (the /recommend request,
    reference src/inference/serve_recommendations.py:213-225). PRIMARY number = HBM-cold: the request runs against a
    rotating set of catalog copies larger than L2 (so neither L2 nor the preceding flush kernel hides anything), one
    request per timed region, launched back to back from the host. Beside it: the same with an L2 flush in front, the
    CUDA-graph replay of DeviceCatalog.topk_small (L2-warm: the serve path keeps hitting the same 76 MB), and the kernel
    alone."""
    import torch

    N, D, k = C2["N"], C2["D"], 10
    g = torch.Generator(device=dev).manual_seed(CATALOG_SEED)
    items = torch.nn.functional.normalize(torch.randn(N, D, device=dev, generator=g), dim=1)
    q = torch.nn.functional.normalize(torch.randn(1, D, device=dev, generator=g), dim=1)
    peaks = _peaks()
    out = {"workload": "C1: batch-1 query x 49,688x384 catalog, top-10 (BASELINE.json configs[0] on the GPU path)", "roofline_bytes": N * D * 4}
    for dt, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        copies = [icr.DeviceCatalog(items.clone(), dtype=dt) for _ in range(4 if dt == torch.float32 else 8)]  # 4 x 76 MB (+ planes) > 126 MB L2
        qd = q.to(dt)
        for c in copies:
            c.topk(qd, k)
        torch.cuda.synchronize()

        def timed(fn, n, pre=None):
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
            for i, (a, b) in enumerate(ev):
                if pre is not None:
                    pre()
                a.record()
                fn(i)
                b.record()
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
            return ts[len(ts) // 2]

        cold_eager = timed(lambda i: copies[i % len(copies)].topk(qd, k), 60)
        flushed = timed(lambda i: copies[0].topk(qd, k), 30, pre=flush.zero_)
        for c in copies:
            c.topk_small(qd, k)
        # the serve path (Recommender._rank) is topk_small: for a device-resident query ONE kernel launch through a prepared
        # argument list. Rotating over the copies keeps the catalog HBM-cold.
        cold = timed(lambda i: copies[i % len(copies)].topk_small(qd, k, copy=False), 60)
        # the same with the host running ahead of the device (a ~40 us spin kernel in front of the start event, as the
        # encoder's kernels are in front of a real request): the device-side time of a request
        cold_dev = timed(lambda i: copies[i % len(copies)].topk_small(qd, k, copy=False), 60, pre=lambda: torch.cuda._sleep(80_000))
        warm = timed(lambda i: copies[0].topk_small(qd, k, copy=False), 60)
        warm_dev = timed(lambda i: copies[0].topk_small(qd, k, copy=False), 60, pre=lambda: torch.cuda._sleep(80_000))
        graphs = [c._graph_for(1, k, ops.PATH_AUTO)[0] for c in copies]  # CUDA-graph form of the request, query already in its input buffer
        cold_replay = timed(lambda i: graphs[i % len(graphs)].replay(), 60)
        warm_replay = timed(lambda i: graphs[0].replay(), 60)
        kt = ops.kernel_timing(lambda: copies[1].topk(qd, k), 20, flush=flush)

        def wall(fn, n=200):  # host wall clock per request, query on the device -> Python lists on the host
            for i in range(10):
                fn(i)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n):
                fn(i)
            return (time.perf_counter() - t0) / n * 1e6

        def two_reads(i):
            v, ix = copies[i % len(copies)].topk_small(qd, k, copy=False)
            return v.tolist(), ix.tolist()

        req_host = wall(lambda i: copies[i % len(copies)].topk_request(qd, k))
        req_two_reads = wall(two_reads)
        nbytes = N * D * (4 if dt == torch.float32 else 2)
        frac = lambda us: nbytes / (us * 1e-6) / 1e9 / peaks["hbm_gbs"]  # noqa: E731
        out[tag] = {"cold_us": cold, "cold_device_us": cold_dev, "cold_graph_replay_us": cold_replay, "cold_eager_call_us": cold_eager,
                    "l2_flushed_us": flushed, "l2_warm_us": warm, "l2_warm_device_us": warm_dev, "graph_replay_us": warm_replay,
                    "kernel_us": kt["ms_per_launch"] * 1e3, "request_to_host_wall_us": req_host, "request_two_device_reads_wall_us": req_two_reads,
                    "hbm_frac_cold": frac(cold), "hbm_frac_cold_device": frac(cold_dev),
                    "hbm_frac_kernel": frac(kt["ms_per_launch"] * 1e3), "catalog_bytes": nbytes}
        del copies
        torch.cuda.empty_cache()
    out["note"] = ("cold_us (primary) = median of 60 requests through DeviceCatalog.topk_small (what Recommender.recommend calls: device query, one "
                   "kernel launch from a prepared argument list), rotating over catalog copies that together exceed L2, CUDA events around each request, "
                   "host launch cost included; cold_device_us = the same with the host running ahead (spin kernel in front of the start event): device-side "
                   "time; cold_graph_replay_us = the request as a CUDA graph, graph.replay() alone; cold_eager_call_us = the rotation through "
                   "DeviceCatalog.topk (generic Python entry: host-bound); l2_flushed_us = one catalog, 512 MB fill before each request (L2 left full of "
                   "dirty lines); l2_warm_* / graph_replay_us = one catalog, L2-warm; kernel_us = the kernel alone, L2 flushed; request_to_host_wall_us = host "
                   "wall clock of DeviceCatalog.topk_request (query on the device -> Python lists on the host: one launch whose last CTA writes "
                   "pinned host memory, one stream sync; cold rotation) and request_two_device_reads_wall_us = the same through topk_small + two "
                   ".tolist() reads; fractions = catalog bytes / time / measured HBM copy peak")
    return out


def bench_c3(icr, ops, dev, flush):
    """BASELINE config 3: MultipleNegativesRankingLoss fwd+bwd, batch 256, dim 384, scale 20, bf16 (reference
    src/training/train_sbert.py:182-185), next to the same loss in PyTorch eager on this GPU."""
    import torch

    B, D, scale = 256, 384, 20.0
    g = torch.Generator(device=dev).manual_seed(7)
    a0 = torch.nn.functional.normalize(torch.randn(B, D, device=dev, generator=g), dim=1)
    p0 = torch.nn.functional.normalize(a0 + 0.3 * torch.randn(B, D, device=dev, generator=g), dim=1)
    res = {"workload": f"C3: MNRL fwd+bwd, B={B}, D={D}, scale={scale:g}"}
    for dt, tag in ((torch.bfloat16, "bf16"), (torch.float32, "f32")):
        a = a0.to(dt).requires_grad_(True)
        p = p0.to(dt).requires_grad_(True)

        def ours():
            a.grad = p.grad = None
            icr.mnrl_loss(a, p, scale).backward()

        def eager():
            a.grad = p.grad = None
            an = torch.nn.functional.normalize(a.float(), dim=1)
            pn = torch.nn.functional.normalize(p.float(), dim=1)
            torch.nn.functional.cross_entropy(an @ pn.T * scale, torch.arange(B, device=dev)).backward()

        def wall(fn, n=200):
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / n * 1e6

        res[tag] = {"fused_us": wall(ours), "eager_us": wall(eager)}
        step = getattr(icr, "mnrl_step_graph", None)
        if step is not None:
            runner = step(B, D, dt, scale, device=dev)
            res[tag]["graph_us"] = wall(lambda: runner(a.detach(), p.detach()))
    res["note"] = "wall clock per step over 200 back-to-back steps (host launch cost included); eager = F.normalize x2 + mm + cross_entropy + autograd on the same GPU"
    return res


def _gen_shard(rows, d, seed, dev, torch):
    """rows x d bf16 unit rows, generated on the device 1M rows at a time (seeded per shard)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    out = torch.empty(rows, d, dtype=torch.bfloat16, device=dev)
    for s0 in range(0, rows, 1 << 20):
        s1 = min(rows, s0 + (1 << 20))
        out[s0:s1] = torch.nn.functional.normalize(torch.randn(s1 - s0, d, device=dev, generator=g), dim=1).to(torch.bfloat16)
    return out


def _witness_topk(q, rows, row_offset, k, torch, chunk=1 << 18):
    """torch fp32 eager on this rank's shard: normalize -> mm -> topk per row block -> merged top-k with global ids."""
    qn = torch.nn.functional.normalize(q.float(), dim=1)
    bv = torch.full((q.shape[0], 0), float("-inf"), device=q.device)
    bi = torch.zeros((q.shape[0], 0), dtype=torch.int64, device=q.device)
    for s in range(0, rows.shape[0], chunk):
        cn = torch.nn.functional.normalize(rows[s : s + chunk].float(), dim=1)
        v, i = torch.topk(qn @ cn.T, min(k, cn.shape[0]), dim=1)
        bv, bi = torch.cat([bv, v], 1), torch.cat([bi, i + s + row_offset], 1)
        if bv.shape[1] > k:
            bv, pos = torch.topk(bv, k, dim=1)
            bi = torch.gather(bi, 1, pos)
    return bv, bi


def bench_sharded(icr, ops, dist, dev, rank, world, flush):
    """STRONG scaling through the collective: the fixed-total catalogs of BASELINE configs 4 and 5, row-sharded over the
    `world` GPUs of this run (world = 1 holds the whole catalog: 15.4 GB and 76.8 GB). Per config and batch size: whole-call
    ms per step (max over ranks, >= 20 steps), the local top-k alone, exchange + merge alone over NVLink peer memory and
    over NCCL, the roofline fraction of the local pass, and `witness_ok`: 16 sampled queries of the merged result against
    torch fp32 eager run on the same shards (scores within 5e-5 relative, ids tie-tolerant)."""
    import torch

    peaks = _peaks()
    k = 100
    configs = [
        {"name": "C4", "total_rows": 10_000_000, "D": 768, "Qs": [1, 64, 1024], "seed": 400},
        {"name": "C5", "total_rows": 100_000_000, "D": 384, "Qs": [4096], "seed": 500},
    ]

    def tmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(fn, n, warm=3):
        for _ in range(warm):
            fn()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(n):
            fn()
        ev1.record()
        barrier()
        return tmax(ev0.elapsed_time(ev1)) / n

    out = {"scaling": "strong (total catalog fixed, rows per GPU = total / n_gpus)", "n_gpus": world, "k": k, "configs": {}}
    peer_error = None
    for cfg in configs:
        total, D = cfg["total_rows"], cfg["D"]
        per = -(-total // world)
        lo, hi = rank * per, min(total, (rank + 1) * per)
        rows = _gen_shard(hi - lo, D, CATALOG_SEED + cfg["seed"] + rank, dev, torch)
        cat = icr.ShardedCatalog(rows, row_offset=lo, total_rows=total, dtype=torch.bfloat16, exchange="peer")
        cat_nccl = cat.with_exchange("nccl")
        g2 = torch.Generator(device=dev).manual_seed(QUERY_SEED + cfg["seed"])
        qall = torch.nn.functional.normalize(torch.randn(max(cfg["Qs"]), D, device=dev, generator=g2), dim=1).to(torch.bfloat16)
        centry = {"total_rows": total, "rows_per_gpu": hi - lo, "D": D, "dtype": "bf16", "shard_bytes": (hi - lo) * D * 2, "batches": {}}
        for Q in cfg["Qs"]:
            q = qall[:Q]
            steps = 20
            e = {"steps": steps}
            use = cat
            if world > 1 and peer_error is None:
                try:
                    cat.topk(q, k)
                except Exception as ex:  # symmetric memory unavailable on this box: every rank takes the NCCL route
                    peer_error = f"{type(ex).__name__}: {ex}"[:300]
            if world > 1:
                flag = torch.tensor([1.0 if peer_error else 0.0], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
                if flag.item() > 0:
                    peer_error = peer_error or "peer exchange failed on another rank"
                    use = cat_nccl
            ms = run(lambda: use.topk(q, k), steps)
            e["ms_per_step"] = ms
            e["queries_per_s"] = Q / (ms * 1e-3)
            e["local_topk_ms"] = run(lambda: cat.local_topk(q, k), steps)
            if world > 1:
                lv, li = cat.local_topk(q, k)
                if use is cat:
                    e["exchange_merge_peer_us"] = run(lambda: cat.exchange_merge(lv, li, k), 50) * 1e3

                    def two_kernels():
                        s_, g_ = cat._peer.all_gather(lv, li)
                        return icr.ops.topk_merge(s_, g_, k)

                    e["exchange_merge_peer_2launch_us"] = run(two_kernels, 50) * 1e3
                    e["fused_launches"] = _launches_of(lambda: cat.topk(q, k), icr)
                e["exchange_merge_nccl_us"] = run(lambda: cat_nccl.exchange_merge(lv, li, k), 50) * 1e3
                e["ms_per_step_nccl"] = run(lambda: cat_nccl.topk(q, k), steps) if use is cat else ms
            # roofline of the local pass: HBM bytes of the shard for small batches, tensor flops for large ones
            flops, nbytes = 2.0 * Q * (hi - lo) * D, (hi - lo) * D * 2
            t = e["local_topk_ms"] * 1e-3
            e["local_tflops"], e["local_gbs"] = flops / t / 1e12, nbytes / t / 1e9
            sustained = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
            ft, fh = e["local_tflops"] / sustained, e["local_gbs"] / peaks["hbm_gbs"]
            e["bound"] = "tensor" if ft > fh else "hbm"
            e["roofline_frac"] = max(ft, fh)
            e["roofline_peak"] = "bf16 sustained" if ft > fh else "hbm copy"
            # witness: 16 sampled queries, torch fp32 eager on the same shards, candidates merged on the host
            sample = torch.arange(0, Q, max(1, Q // 16), device=dev)[:16]
            v, i = use.topk(q, k)
            wv, wi = _witness_topk(q[sample], rows, lo, k, torch)
            if world > 1:
                gv = [torch.empty_like(wv) for _ in range(world)]
                gi = [torch.empty_like(wi) for _ in range(world)]
                dist.all_gather(gv, wv)
                dist.all_gather(gi, wi)
                wv, wi = torch.cat(gv, 1), torch.cat(gi, 1)
                wv, pos = torch.topk(wv, k, dim=1)
                wi = torch.gather(wi, 1, pos)
            order = torch.argsort(wv, dim=1, descending=True, stable=True)
            wv, wi = torch.gather(wv, 1, order), torch.gather(wi, 1, order)
            sv, si = v[sample], i[sample]
            denom = wv.abs().clamp_min(0.05)
            rel = ((sv - wv).abs() / denom).max().item()
            gap_ok = torch.ones_like(wv, dtype=torch.bool)
            tol = 1e-4 * denom  # ids are only held where the witness's neighbouring scores are further apart than this
            gap_ok[:, 1:] &= (wv[:, :-1] - wv[:, 1:]) > tol[:, 1:]
            gap_ok[:, :-1] &= (wv[:, :-1] - wv[:, 1:]) > tol[:, :-1]
            gap_ok[:, -1] = False
            mism = int(((si != wi) & gap_ok).sum().item())
            e["witness_max_rel_err"] = rel
            e["witness_id_mismatch"] = mism
            e["witness_ok"] = bool(rel <= 5e-5 and mism == 0 and bool(((i >= 0) & (i < total)).all().item()))
            centry["batches"][f"Q{Q}"] = e
        out["configs"][cfg["name"]] = centry
        del cat, cat_nccl, rows, qall
        torch.cuda.empty_cache()
    out["exchange"] = ("NCCL all-gather of packed candidates + device merge (peer exchange unavailable)" if peer_error else
                       "icr_cos_topk_sharded: shard search + NVLink peer-memory push + flags + merge in one library call (one launch for Q <= 7: the "
                       "exchange and merge run in the tail of the GEMV kernel; otherwise the search, then ONE exchange+merge kernel); "
                       "the round-1 two-launch exchange and the NCCL route timed beside it") if world > 1 else "none (one GPU holds the whole catalog)"
    out["peer_exchange_error"] = peer_error
    out["witness"] = "torch fp32 eager (normalize -> mm -> topk) on the same bf16 shards, 16 sampled queries per batch size, per-rank top-k gathered and merged"
    out["oracle_ok"] = all(b["witness_ok"] for c in out["configs"].values() for b in c["batches"].values())
    return out


def _launches_of(fn, icr):
    fn()
    return int(icr.ops.last_launch_count())


if __name__ == "__main__":
    main()
