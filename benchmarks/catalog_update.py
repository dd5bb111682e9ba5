"""Times in-place catalog changes against a full rebuild (CUDA events; every timed call ends in a device synchronise).

Shapes: C2 (49,688 x 384, the reference's corpus) for each catalog dtype, and a 2M x 768 bf16 catalog (C4-like). Per shape:
  - update_rows for M in {1, 16, 256, 4096} rows (scattered);
  - append_rows(1000): the first append (which reallocates with headroom) and a second one inside the reserve;
  - remove_rows of 1,000 scattered rows;
  - a full rebuild (DeviceCatalog over a device-resident fp32 matrix).
Each timing is the median of `--reps` calls after one warm-up call. The card's name and power limit are read in the same run.

    python benchmarks/catalog_update.py [--reps 5] [--out profiles/r06_catalog_updates.txt]
"""

from __future__ import annotations

import argparse
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import instacart_next_order_recommendation_b200 as icr  # noqa: E402


def _ms(fn, reps):
    times = []
    for _ in range(reps + 1):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    times = sorted(times[1:] if reps else times)
    return times[len(times) // 2]


def bench_shape(name, N, D, dtype, reps, lines):
    g = torch.Generator(device="cuda").manual_seed(N + D)
    X = F.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    rebuild = _ms(lambda: icr.DeviceCatalog(X, dtype=dtype), reps)
    cat = icr.DeviceCatalog(X.clone(), dtype=dtype)
    row = [f"{name:<22} rebuild {rebuild:9.3f} ms"]
    for M in (1, 16, 256, 4096):
        rows = torch.randperm(N, device="cuda", generator=g)[:M].cpu()
        Y = torch.randn(M, D, device="cuda", generator=g)
        row.append(f"update M={M:<4} {_ms(lambda: cat.update_rows(rows, Y), reps):8.3f} ms")
    A = torch.randn(1000, D, device="cuda", generator=g)
    first = []

    def grow():  # a fresh catalog per call: each call is a first append, which reallocates
        c = icr.DeviceCatalog(X.clone(), dtype=dtype)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        c.append_rows(A)
        e.record()
        torch.cuda.synchronize()
        first.append(s.elapsed_time(e))

    for _ in range(reps + 1):
        grow()
    realloc = sorted(first[1:])[len(first[1:]) // 2]
    cat.append_rows(A)  # reserve 1.5 N: the appends below stay inside it
    inside = _ms(lambda: cat.append_rows(A), reps)
    row.append(f"append 1000 realloc {realloc:8.3f} ms  in-reserve {inside:8.3f} ms")
    n = len(cat)
    removes = []
    for _ in range(reps + 1):
        gone = torch.randperm(n, generator=torch.Generator().manual_seed(len(removes)))[:1000].tolist()
        removes.append(_ms(lambda: cat.remove_rows(gone), 0))
        n = len(cat)
    row.append(f"remove 1000 {sorted(removes[1:])[len(removes[1:]) // 2]:8.3f} ms")
    lines.append("  ".join(row[:1]) + "\n    " + "\n    ".join(row[1:]))
    del cat, X
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles/r06_catalog_updates.txt")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    lines = [f"# in-place catalog changes vs full rebuild; median of {args.reps} calls, CUDA events, synchronised",
             f"# card: {card}", f"# torch {torch.__version__}"]
    for name, N, D, dtype in (("c2_fp32", 49_688, 384, torch.float32), ("c2_bf16", 49_688, 384, torch.bfloat16),
                              ("c2_fp16", 49_688, 384, torch.float16), ("c2_int8", 49_688, 384, torch.int8),
                              ("2M_x_768_bf16", 2_000_000, 768, torch.bfloat16)):
        bench_shape(name, N, D, dtype, args.reps, lines)
        print(lines[-1], flush=True)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text("\n".join(lines) + "\n")
    print(f"wrote {out}")


if __name__ == "__main__":
    main()
