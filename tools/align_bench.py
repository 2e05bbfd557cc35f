#!/usr/bin/env python
"""Developer timing of K8 (gfx_align) on one B200, next to the host NumPy DP
(oracle/align_oracle.py) that a user runs today on embeddings copied back.

    python tools/align_bench.py [N]        the first N shapes
    python tools/align_bench.py --quick    every shape with 1/100 of the pairs, one repeat
    python tools/align_bench.py --out F    also write the rows to F as one JSON list

Tables are random unit fp16 rows (a 200k-row query table and a 400k-row target
table, 154 MB: larger than the 126 MB L2), and each pair takes random segment
starts in them.  The timed region is gfx_align alone (the kernel and its finish
kernel) on pairs already validated and resident on the device; align_pairs adds
its host validation on top.  Each repeat is a window of at least 0.5 s of back-to-
back calls after a warm-up call; five repeats give the spread.

Rates: useful cells/s counts q_len * t_len per pair (GCUPS), useful TFLOP/s the
2 * 128 FLOP of the dot product of each such cell.  The host rate is the float32
NumPy oracle (S by one matmul, then the anti-diagonal DP) on a sample of the
shape's pairs.  Card name, power limit and maximum SM clock are read in the same
call.  Each shape's row is printed as one JSON line."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from ginfinity_b200 import _native as nat  # noqa: E402
from oracle.align_oracle import align_fp32  # noqa: E402

PARAMS = (0.05, 0.5, 0.1)          # offset, gap_open, gap_extend
Q_ROWS, T_ROWS = 200_000, 400_000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return {"card": torch.cuda.get_device_name(0), "nvidia_smi": out}


def unit(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(n, 128, generator=g, device="cuda")
    return (a / a.norm(dim=1, keepdim=True)).half()


def shapes(quick):
    scale = 100 if quick else 1
    rng = np.random.default_rng(0)
    P = 100_000 // scale
    mixed = np.exp(rng.uniform(np.log(16), np.log(4096), size=(P, 2))).astype(np.int64)
    return [
        ("64x64", np.full((1_000_000 // scale, 2), 64)),
        ("128x128", np.full((1_000_000 // scale, 2), 128)),
        ("200x400", np.tile([200, 400], (200_000 // scale, 1))),
        ("2000x4000", np.tile([2000, 4000], (256, 1))),
        ("mixed_16_4096_loguniform", mixed),
    ]


def make_pairs(lens, rng):
    P = len(lens)
    qs = rng.integers(0, Q_ROWS - lens[:, 0] + 1, size=P)
    ts = rng.integers(0, T_ROWS - lens[:, 1] + 1, size=P)
    return np.stack([qs, lens[:, 0], ts, lens[:, 1]], 1).astype(np.int64)


def host_rate(Qh, Th, pairs, budget_s=3.0):
    cells, t0 = 0, time.perf_counter()
    for qs, ql, ts, tl in pairs:
        S = Qh[qs:qs + ql].astype(np.float32) @ Th[ts:ts + tl].astype(np.float32).T
        align_fp32(S, *PARAMS)
        cells += int(ql) * int(tl)
        if time.perf_counter() - t0 > budget_s:
            break
    return cells / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("count", nargs="?", type=int)
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", type=Path, help="write the rows here as one JSON list")
    args = ap.parse_args()
    info = card()
    Q, T = unit(Q_ROWS, 1), unit(T_ROWS, 2)
    Qh, Th = Q.cpu().numpy(), T.cpu().numpy()
    stream = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(1)
    rows = []
    todo = shapes(args.quick)[:args.count] if args.count else shapes(args.quick)
    for name, lens in todo:
        pairs = make_pairs(lens, rng)
        P = len(pairs)
        multi = pairs[:, 1] > 128
        max_t = int(pairs[multi, 3].max()) if multi.any() else 0
        pd = torch.from_numpy(pairs).cuda()
        score = torch.empty(P, dtype=torch.float32, device="cuda")
        coords = torch.empty((P, 4), dtype=torch.int32, device="cuda")
        need = nat.lib.gfx_align_workspace_bytes(P, max_t)
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")

        def call():
            nat.check(nat.lib.gfx_align(Q.data_ptr(), Q_ROWS, T.data_ptr(), T_ROWS, pd.data_ptr(), P,
                                        *PARAMS, score.data_ptr(), coords.data_ptr(), ws.data_ptr(),
                                        need, stream))

        call()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        call()
        b.record()
        torch.cuda.synchronize()
        once = a.elapsed_time(b) * 1e-3
        iters = max(1, int(np.ceil(0.5 / max(once, 1e-6))))
        seconds = []
        for _ in range(1 if args.quick else 5):
            a.record()
            for _ in range(iters):
                call()
            b.record()
            torch.cuda.synchronize()
            seconds.append(a.elapsed_time(b) * 1e-3 / iters)
        cells = float((pairs[:, 1] * pairs[:, 3]).sum())
        t = float(np.median(seconds))
        sample = pairs[rng.permutation(P)[:200]]
        host = host_rate(Qh, Th, sample)
        row = {"shape": name, "pairs": P, "useful_cells": cells, "calls_per_window": iters,
               "seconds_median": t, "seconds_min": min(seconds), "seconds_max": max(seconds),
               "gcups": cells / t / 1e9, "gcups_min": cells / max(seconds) / 1e9,
               "gcups_max": cells / min(seconds) / 1e9, "useful_tflops": 256 * cells / t / 1e12,
               "pairs_per_s": P / t, "host_numpy_gcups": host / 1e9,
               "speedup_over_host": cells / t / host, "params": PARAMS, **info}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del pd, score, coords, ws
        torch.cuda.empty_cache()
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(rows, indent=1))


if __name__ == "__main__":
    main()
