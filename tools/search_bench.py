#!/usr/bin/env python
"""Developer timing of K5 (gfx_topk) on one B200: TFLOP/s of the fused
GEMM + top-k scan at a few shapes, next to torch.matmul + torch.topk on the
same inputs (library bar).  Prints and writes gpurun_out/search.json -- unless
SEARCH_BENCH_NO_JSON is set: round 1's tools/gpu_round.sh re-ran this very
command under `ncu --set full` (to capture topk_scan), and that second run
overwrote search.json with timings whose event-bracketed region contained
ncu's kernel replays (the "14.6 s / 41.8 s cosine" rows of
profiles/r01_d/f_search_timing.json).  A run under a profiler must not write
the timing file.

    python tools/search_bench.py [N]                 fp16 rows, the first N shapes
    python tools/search_bench.py --dtype float32     fp32 rows (gfx_topk_f32) and,
        from the same call and data rounded to fp16, fp16 rows beside them
        (every row of such a run carries its "dtype")

Issued TFLOP/s counts the tensor work the scan does (three fp16 products per
fp32 product for float32 rows), useful TFLOP/s one product per (query, row)
pair.  The card's name and power limit are recorded with the rows."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from ginfinity_b200 import _native as nat  # noqa: E402
from ginfinity_b200.search import EmbeddingIndex  # noqa: E402


def unit(n, seed, dtype=torch.float16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(n, 128, generator=g, device="cuda")
    return (a / a.norm(dim=1, keepdim=True)).to(dtype)


def timed(fn, iters=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(True), torch.cuda.Event(True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3


def card():
    """Name and power limit of cuda:0, read in the same call as the timings."""
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"card": torch.cuda.get_device_name(0), "power_limit": limit}


def time_search(index, q, metric, D):
    nat.profile_enable("topk")
    t = timed(lambda: index.search(q, 10, metric), iters=2 if D > 5_000_000 else 3)
    nat.profile_enable()
    nat.profile_read("topk")
    return t


def main_fp16(shapes):
    out = []
    for Q, D in shapes:
        q, db = unit(Q, 1), unit(D, 2)
        index = EmbeddingIndex(db, device="cuda")
        for metric in ("cosine", "l2"):
            t = time_search(index, q, metric, D)
            flop = 2.0 * 128 * Q * D
            row = {"Q": Q, "D": D, "metric": metric, "seconds": t, "tflops": flop / t / 1e12,
                   "db_rows_per_s": D / t, "fallbacks": index.last_fallbacks()}
            if Q * D <= 4096 * 1_000_000:
                def lib():
                    s = q @ db.T
                    return s.topk(10, dim=1)
                row["torch_matmul_topk_seconds"] = timed(lib)
            print(row, flush=True)
            out.append(row)
        del index, db
        torch.cuda.empty_cache()
    return out


def main_fp32(shapes):
    """fp32 rows, then the same rows rounded to fp16, per shape and metric."""
    out, info = [], card()
    for Q, D in shapes:
        q32, db32 = unit(Q, 1, torch.float32), unit(D, 2, torch.float32)
        for dtype in ("float32", "float16"):
            q, db = (q32, db32) if dtype == "float32" else (q32.half(), db32.half())
            index = EmbeddingIndex(db, device="cuda")
            for metric in ("cosine", "l2"):
                t = time_search(index, q, metric, D)
                useful = 2.0 * 128 * Q * D
                issued = useful * (3 if dtype == "float32" else 1)
                row = {"dtype": dtype, "Q": Q, "D": D, "metric": metric, "seconds": t,
                       "issued_tflops": issued / t / 1e12, "useful_tflops": useful / t / 1e12,
                       "fallbacks": index.last_fallbacks(), **info}
                print(row, flush=True)
                out.append(row)
            del index, q, db
            torch.cuda.empty_cache()
        del q32, db32
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shapes", nargs="?", type=int, help="run the first N shapes only")
    ap.add_argument("--dtype", choices=("float16", "float32"), default="float16")
    args = ap.parse_args()
    if args.dtype == "float32":
        shapes = [(100_000, 1_000_000), (4096, 1_000_000), (100_000, 12_500_000)]
    else:
        shapes = [(4096, 1_000_000), (100_000, 1_000_000), (100_000, 12_500_000)]
    if args.shapes:
        shapes = shapes[:args.shapes]
    out = main_fp32(shapes) if args.dtype == "float32" else main_fp16(shapes)
    import os
    if os.environ.get("SEARCH_BENCH_NO_JSON"):
        return
    (ROOT / "gpurun_out").mkdir(exist_ok=True)
    (ROOT / "gpurun_out" / "search.json").write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
