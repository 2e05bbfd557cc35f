#!/usr/bin/env python
"""Developer timing of K5 (gfx_topk) on one B200: TFLOP/s of the fused
GEMM + top-k scan at a few shapes, next to torch.matmul + torch.topk on the
same inputs (library bar).  Prints and writes gpurun_out/search.json -- unless
SEARCH_BENCH_NO_JSON is set: round 1's tools/gpu_round.sh re-ran this very
command under `ncu --set full` (to capture topk_scan), and that second run
overwrote search.json with timings whose event-bracketed region contained
ncu's kernel replays (the "14.6 s / 41.8 s cosine" rows of
profiles/r01_d/f_search_timing.json).  A run under a profiler must not write
the timing file."""
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from ginfinity_b200 import _native as nat  # noqa: E402
from ginfinity_b200.search import EmbeddingIndex  # noqa: E402


def unit(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(n, 128, generator=g, device="cuda")
    return (a / a.norm(dim=1, keepdim=True)).half()


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


def main():
    shapes = [(4096, 1_000_000), (100_000, 1_000_000), (100_000, 12_500_000)]
    if len(sys.argv) > 1:
        shapes = shapes[:int(sys.argv[1])]
    out = []
    for Q, D in shapes:
        q, db = unit(Q, 1), unit(D, 2)
        index = EmbeddingIndex(db, device="cuda")
        for metric in ("cosine", "l2"):
            nat.profile_enable("topk")
            t = timed(lambda: index.search(q, 10, metric), iters=2 if D > 5_000_000 else 3)
            nat.profile_enable()
            nat.profile_read("topk")
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
    import os
    if os.environ.get("SEARCH_BENCH_NO_JSON"):
        return
    (ROOT / "gpurun_out").mkdir(exist_ok=True)
    (ROOT / "gpurun_out" / "search.json").write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
