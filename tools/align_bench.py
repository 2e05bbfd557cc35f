#!/usr/bin/env python
"""Developer timing of K8 (gfx_align) on one B200, next to the host NumPy DP
(oracle/align_oracle.py) that a user runs today on embeddings copied back.

    python tools/align_bench.py [N]        the first N shapes
    python tools/align_bench.py --quick    every shape with 1/100 of the pairs, one repeat
    python tools/align_bench.py --out F    also write the rows to F as one JSON list
    python tools/align_bench.py --traceback [--quick] [--out F]
                                           the traceback (align_paths) instead, below

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
call.  Each shape's row is printed as one JSON line.

--traceback runs every shape in two regimes: "random" (the tables above; boxes
are small) and "planted" (targets from a noisy copy of the query table, each
pair's target holding its query at a random shift; a box is most of the pair).
For each it reports
  * the box DP pass: cells of the boxes per second of the trace DP kernel
    (align_kernel<true>), and that rate over the score kernel's
    (align_kernel<false>) on the same boxes;
  * the walk: path steps per second of align_walk_kernel, and microseconds per
    pair;
  * align_paths against align_pairs end to end (host clock around the call and a
    device synchronise; median of three).
Kernel times come from torch.profiler over three calls of each, after a warm-up
call, in their own profiling window; the end-to-end times are taken with the
profiler off."""
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


def kernel_ms(fn, calls=3):
    """Mean device milliseconds per call of each align kernel launched by fn()."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for key in ("align_kernel<true>", "align_kernel<false>", "align_walk_kernel", "align_code_offsets_kernel",
                    "align_finish_kernel"):
            if key in e.key:
                out[key] = out.get(key, 0.0) + e.device_time_total / 1e3 / calls
    return out


def wall(fn, repeats=3):
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return float(np.median(times))


def traceback_rows(args, info):
    from ginfinity_b200 import align as al
    Q, T = unit(Q_ROWS, 1), unit(T_ROWS, 2)
    g = torch.Generator(device="cuda").manual_seed(3)
    noisy = Q.float() + 0.3 * torch.randn(Q.shape, generator=g, device="cuda") / np.sqrt(128)
    Tn = (noisy / noisy.norm(dim=1, keepdim=True)).half()
    del noisy
    stream = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(1)
    kw = dict(offset=PARAMS[0], gap_open=PARAMS[1], gap_extend=PARAMS[2])
    rows = []
    todo = shapes(args.quick)[:args.count] if args.count else shapes(args.quick)
    for name, lens in todo:
        for regime in ("random", "planted"):
            if regime == "random":
                pairs, tq, tt = make_pairs(lens, rng), Q, T
            else:
                P = len(lens)
                ql, tl = lens[:, 0], lens[:, 1]
                qs = rng.integers(4096, Q_ROWS - 4096 - ql + 1, size=P)
                ts = qs - rng.integers(0, np.maximum(tl - ql, 0) + 1)
                pairs, tq, tt = np.stack([qs, ql, ts, tl], 1).astype(np.int64), Q, Tn
            P = len(pairs)
            pd = torch.from_numpy(pairs).cuda()
            res, paths = al.align_paths(tq, tt, pd, **kw)
            qb, qe, tb, te = torch.stack(res[1:], 1).cpu().numpy().astype(np.int64).T
            has = qb >= 0
            h, w = np.where(has, qe - qb, 0), np.where(has, te - tb, 0)
            boxes = np.stack([pairs[:, 0] + np.maximum(qb, 0), h, pairs[:, 2] + np.maximum(tb, 0), w], 1)
            bd = torch.from_numpy(boxes).cuda()
            box_cells = float((h * w).sum())
            steps = float(paths.lengths.sum().item())
            score = torch.empty(P, dtype=torch.float32, device="cuda")
            coords = torch.empty((P, 4), dtype=torch.int32, device="cuda")
            multi = h > 128
            need_s = nat.lib.gfx_align_workspace_bytes(P, int(w[multi].max()) if multi.any() else 0)
            ws_s = torch.empty(need_s, dtype=torch.uint8, device="cuda")
            code_bytes = int((h * ((w + 31) // 32) * 16).sum())
            need_t = nat.lib.gfx_align_trace_workspace_bytes(P, code_bytes)
            ws_t = torch.empty(need_t, dtype=torch.uint8, device="cuda")
            cap = np.maximum(h + w - 1, 0)
            od = torch.from_numpy(np.concatenate([[0], np.cumsum(cap)[:-1]]).astype(np.int64)).cuda()
            ops = torch.empty(max(int(cap.sum()), 1), dtype=torch.uint8, device="cuda")
            lens_d = torch.empty(P, dtype=torch.int32, device="cuda")

            def score_boxes():
                nat.check(nat.lib.gfx_align(tq.data_ptr(), len(tq), tt.data_ptr(), len(tt), bd.data_ptr(), P,
                                            *PARAMS, score.data_ptr(), coords.data_ptr(), ws_s.data_ptr(),
                                            need_s, stream))

            def trace_boxes():
                nat.check(nat.lib.gfx_align_trace(tq.data_ptr(), len(tq), tt.data_ptr(), len(tt), bd.data_ptr(),
                                                  P, *PARAMS, score.data_ptr(), coords.data_ptr(),
                                                  ops.data_ptr(), od.data_ptr(), lens_d.data_ptr(),
                                                  ws_t.data_ptr(), need_t, stream))

            ks = kernel_ms(score_boxes)
            kt = kernel_ms(trace_boxes)
            assert (lens_d.cpu() == paths.lengths.cpu()).all()
            del ws_s, ws_t, ops
            t_pairs = wall(lambda: al.align_pairs(tq, tt, pd, **kw))
            t_paths = wall(lambda: al.align_paths(tq, tt, pd, **kw))
            score_ms, trace_ms = ks.get("align_kernel<false>", 0.0), kt.get("align_kernel<true>", 0.0)
            walk_ms = kt.get("align_walk_kernel", 0.0)
            row = {"shape": name, "regime": regime, "pairs": P, "pair_cells": float((pairs[:, 1] * pairs[:, 3]).sum()),
                   "box_cells": box_cells, "aligned_pairs": int(has.sum()), "path_steps": steps,
                   "score_kernel_on_boxes_ms": score_ms, "trace_kernel_on_boxes_ms": trace_ms,
                   "box_gcups_score": box_cells / score_ms / 1e6 if score_ms else None,
                   "box_gcups_trace": box_cells / trace_ms / 1e6 if trace_ms else None,
                   "trace_over_score_rate": score_ms / trace_ms if trace_ms else None,
                   "offsets_kernel_ms": kt.get("align_code_offsets_kernel", 0.0),
                   "walk_ms": walk_ms, "walk_steps_per_s": steps / walk_ms * 1e3 if walk_ms else None,
                   "walk_us_per_pair": walk_ms * 1e3 / P,
                   "align_pairs_s": t_pairs, "align_paths_s": t_paths, "paths_over_pairs": t_paths / t_pairs,
                   "params": PARAMS, **info}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del pd, bd, score, coords, res, paths
            torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("count", nargs="?", type=int)
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--traceback", action="store_true", help="time align_paths and its kernels instead")
    ap.add_argument("--out", type=Path, help="write the rows here as one JSON list")
    args = ap.parse_args()
    info = card()
    if args.traceback:
        rows = traceback_rows(args, info)
        if args.out is not None:
            args.out.parent.mkdir(parents=True, exist_ok=True)
            args.out.write_text(json.dumps(rows, indent=1))
        return
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
