"""Local alignment of per-nucleotide embeddings (Smith-Waterman, affine gaps)
on the GPU: K8 of libgfx.so (csrc/gfx_align.cu).  `align_pairs` gives each
pair's score and region, `align_paths` also the aligned path.

The reference ships scoring parameters for a separate aligner
(`alignment-config`, src/ginfinity/api.py:47-50) but not the aligner, so the
contract below is this package's own.  `align_pairs` does not read
`alignment.json`: which of its keys would map onto which parameter here is not
known, so every parameter is given explicitly and none has a default.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import numpy as np
import torch

from . import _native as nat
from .records import MAXIMUM_LENGTH_NT

DIM = 128
MAX_SEGMENT = MAXIMUM_LENGTH_NT
# align_paths: bytes of DP pointer record per gfx_align_trace call (4 bits per cell of the boxes
# in the call).  One 4096 x 4096 box takes 8 MiB, so a single box always fits.
CODE_BUDGET = 1 << 30


class Alignments(NamedTuple):
    """One entry per pair, all on the device.  Coordinates are half-open and
    relative to the pair's segments; a pair without a positive cell has score
    0 and coordinates -1."""
    score: torch.Tensor          # float32 [P]
    query_begin: torch.Tensor    # int32 [P]
    query_end: torch.Tensor
    target_begin: torch.Tensor
    target_end: torch.Tensor


def align_pairs(queries, targets, pairs, *, offset: float, gap_open: float,
                gap_extend: float, device=None) -> Alignments:
    """Best local alignment of each pair of embedding segments.

    `queries` [Nq, 128] and `targets` [Nt, 128] are float16 tables (they may be
    the same tensor).  CUDA tensors are used in place; NumPy arrays and CPU
    tensors are copied to `device` (default: the tables' CUDA device, else the
    current one).  `pairs` int64 [P, 4] holds rows (q_start, q_len, t_start,
    t_len): rows q_start .. q_start+q_len-1 of `queries` against rows
    t_start .. t_start+t_len-1 of `targets`, each length 0..4096 and inside its
    table.

    For query row i and target row j of a pair, in fp32 in this order:

        S(i,j) = q_i . t_j       tensor cores, fp16 inputs, fp32 accumulation
        s      = S(i,j) - offset
        E(i,j) = max(H(i,j-1) - gap_open, E(i,j-1) - gap_extend)
        F(i,j) = max(H(i-1,j) - gap_open, F(i-1,j) - gap_extend)
        H(i,j) = max(0, H(i-1,j-1) + s, E(i,j), F(i,j))

    with H = 0 and E, F = -inf outside the segments: a gap of length L costs
    gap_open + (L-1) * gap_extend.  The score is the largest H; ties of the
    end cell go to the smaller i, then the smaller j.  A positive H takes its
    start from the first of diagonal, E, F that attains it (opening beats
    extending), and a diagonal step from H = 0 starts the alignment there.

    Accuracy: S is the tensor-core sum, within 2^-14 |q_i| |t_j| of the exact
    dot product, so the score is within min(q_len, t_len) * 2^-14 * max|q| *
    max|t| of the float64 optimum, plus the fp32 rounding of the DP.  Results
    are bit-reproducible: a pair gives the same bits in any batch, at any
    position and table offset.

    Validation reads `pairs` and checks every table component is finite on
    the host: one host synchronisation when `pairs` or the tables are on the
    device.  Everything else is enqueued on the current stream.

    Device-resident route, an all-core shard encoded in HBM::

        ds = DeviceShard.from_shard(shard, "cuda")
        emb = encoder.encode_device_shard(ds)              # [N, 128] float16
        ptr = ds.node_ptr.cpu()
        a, b = 3, 7                                        # records to align
        pairs = torch.tensor([[ptr[a], ptr[a+1] - ptr[a], ptr[b], ptr[b+1] - ptr[b]]])
        res = align_pairs(emb, emb, pairs, offset=..., gap_open=..., gap_extend=...)

    Host route, from `encode_many` arrays::

        embs = encoder.encode_many(records)                # list of [L, 128] float16
        table = np.concatenate(embs)
        ptr = np.concatenate([[0], np.cumsum([len(e) for e in embs])])

    Float32 embeddings are not supported; cast them to float16.
    """
    score, coords = _score_pass(_prepare(queries, targets, pairs, offset, gap_open, gap_extend, device))
    return Alignments(score, *coords.unbind(1))


class AlignmentPaths(NamedTuple):
    """The aligned path of each pair, on the device.  Pair p's path is
    ops[offsets[p] : offsets[p] + lengths[p]], one op per step from
    (query_begin, target_begin) to (query_end - 1, target_end - 1):
    0 = M (query row with target row), 1 = I (query row with a gap),
    2 = D (target row with a gap)."""
    ops: torch.Tensor            # uint8
    offsets: torch.Tensor        # int64 [P]
    lengths: torch.Tensor        # int32 [P]

    def cigars(self) -> list:
        """SAM-style run-length strings, one per pair ("12M2I30M1D5M"; "" for a
        pair without an alignment), from one device-to-host copy."""
        P = len(self.lengths)
        buf = torch.cat([self.offsets.to(torch.int64).contiguous().view(torch.uint8),
                         self.lengths.to(torch.int32).contiguous().view(torch.uint8),
                         self.ops.reshape(-1).view(torch.uint8)]).cpu().numpy()
        offsets = buf[:8 * P].view(np.int64)
        lengths = buf[8 * P:12 * P].view(np.int32)
        ops = buf[12 * P:]
        out = []
        for o, n in zip(offsets.tolist(), lengths.tolist()):
            path = ops[o:o + n]
            if n <= 0:
                out.append("")
                continue
            ends = np.flatnonzero(np.diff(path)).tolist() + [n - 1]
            begin, parts = 0, []
            for e in ends:
                parts.append(f"{e - begin + 1}{'MID'[path[e]]}")
                begin = e + 1
            out.append("".join(parts))
        return out


def align_paths(queries, targets, pairs, *, offset: float, gap_open: float,
                gap_extend: float, device=None) -> tuple:
    """`align_pairs` and the aligned path of every pair: (Alignments,
    AlignmentPaths).  Arguments, validation and errors are those of
    `align_pairs`, and the Alignments are the same bits.

    The path is the one the tie rules of `align_pairs` define: followed back
    from the end cell, H takes the first of diagonal, E, F that attains it, E
    and F prefer opening to extending, and a diagonal step from H = 0 is the
    start.  It starts and ends with M; #M + #I = query_end - query_begin and
    #M + #D = target_end - target_begin.  A pair with score 0 has an empty
    path.  Rescoring the path in fp32 gives the score bit for bit: v = 0 + s
    at the first M, then + s per M, - gap_open per gap opened (after M or
    after the other gap kind), - gap_extend per gap extended.

    How: after the score pass the coordinates come back to the host (16 bytes
    per pair, one synchronisation).  The DP then runs again over each pair's
    box [query_begin, query_end) x [target_begin, target_end) only, recording
    4 bits per cell, and a walk follows them back from the box's corner.
    Inside the box every value is at most its value in the whole segments and
    equal along the path, so the box pass must return the same score at
    (0, h, 0, w); a pair where it does not raises RuntimeError (a library
    bug, never a wrong path).  Boxes run in calls of at most CODE_BUDGET
    bytes of pointer record.
    """
    pr = _prepare(queries, targets, pairs, offset, gap_open, gap_extend, device)
    score, coords = _score_pass(pr)
    dev, P = pr.dev, len(pr.pairs)
    lengths = torch.zeros(P, dtype=torch.int32, device=dev)
    if P == 0:
        return (Alignments(score, *coords.unbind(1)),
                AlignmentPaths(torch.empty(0, dtype=torch.uint8, device=dev),
                               torch.empty(0, dtype=torch.int64, device=dev), lengths))
    qb, qe, tb, te = coords.cpu().numpy().astype(np.int64).T
    has = qb >= 0
    h, w = np.where(has, qe - qb, 0), np.where(has, te - tb, 0)
    boxes = np.stack([pr.pairs[:, 0] + np.maximum(qb, 0), h, pr.pairs[:, 2] + np.maximum(tb, 0), w], 1)
    want = np.where(has[:, None], np.stack([np.zeros(P, np.int64), h, np.zeros(P, np.int64), w], 1), -1)
    cap = np.maximum(h + w - 1, 0)
    offsets = np.concatenate([[0], np.cumsum(cap)[:-1]]).astype(np.int64)
    total = int(cap.sum())
    code_end = np.cumsum(h * ((w + 31) // 32) * 16)
    boxes_dev = torch.from_numpy(boxes.astype(np.int64)).to(dev, non_blocking=True)
    want_dev = torch.from_numpy(want.astype(np.int32)).to(dev, non_blocking=True)
    offsets_dev = torch.from_numpy(offsets).to(dev, non_blocking=True)
    ops = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
    box_score = torch.empty(P, dtype=torch.float32, device=dev)
    box_coords = torch.empty((P, 4), dtype=torch.int32, device=dev)
    go, ge, th = pr.params
    q, t = pr.q, pr.t
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        a = 0
        while a < P:
            done = int(code_end[a - 1]) if a else 0
            b = max(int(np.searchsorted(code_end, done + CODE_BUDGET, side="right")), a + 1)
            need = nat.lib.gfx_align_trace_workspace_bytes(b - a, int(code_end[b - 1]) - done)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            nat.check(nat.lib.gfx_align_trace(
                q.data_ptr() if len(q) else None, len(q), t.data_ptr() if len(t) else None, len(t),
                boxes_dev[a:].data_ptr(), b - a, th, go, ge, box_score[a:].data_ptr(),
                box_coords[a:].data_ptr(), ops.data_ptr(), offsets_dev[a:].data_ptr(),
                lengths[a:].data_ptr(), ws.data_ptr(), need, stream))
            a = b
    bad = ((box_score.view(torch.int32) != score.view(torch.int32)) | (box_coords != want_dev).any(1)
           | (lengths < 0))
    if bool(bad.any()):
        p = int(torch.nonzero(bad)[0])
        raise RuntimeError(
            f"align_paths: pair {p}: the pass over its box [{int(boxes[p, 0])}, +{int(h[p])}) x "
            f"[{int(boxes[p, 2])}, +{int(w[p])}) gave score {float(box_score[p])} at "
            f"{tuple(int(v) for v in box_coords[p].tolist())}, path length {int(lengths[p])}; the score "
            f"pass gave {float(score[p])}")
    return Alignments(score, *coords.unbind(1)), AlignmentPaths(ops[:total], offsets_dev, lengths)


class _Problem(NamedTuple):
    q: torch.Tensor
    t: torch.Tensor
    pairs: np.ndarray            # int64 [P, 4], host
    pairs_dev: torch.Tensor
    max_t: int
    params: list                 # gap_open, gap_extend, offset as float32 values
    dev: torch.device


def _prepare(queries, targets, pairs, offset, gap_open, gap_extend, device) -> _Problem:
    go, ge, th = _parameters(offset, gap_open, gap_extend)
    q = _table(queries, "queries")
    t = q if targets is queries else _table(targets, "targets")
    pairs_host, max_t = _pairs(pairs, len(q), len(t))
    for name, table in (("queries", q), ("targets", t)):
        if not _all_finite(table):
            raise ValueError(f"{name} holds a non-finite component")
    dev = _device(device, queries, targets)
    q = q.to(dev, non_blocking=True).contiguous()
    t = q if targets is queries else t.to(dev, non_blocking=True).contiguous()
    pairs_dev = None
    if len(pairs_host):
        if isinstance(pairs, torch.Tensor) and pairs.device == dev:
            pairs_dev = pairs.to(torch.int64).contiguous()
        else:
            pairs_dev = torch.from_numpy(pairs_host).to(dev, non_blocking=True)
    return _Problem(q, t, pairs_host, pairs_dev, max_t, [go, ge, th], dev)


def _score_pass(pr: _Problem):
    q, t, P, dev = pr.q, pr.t, len(pr.pairs), pr.dev
    go, ge, th = pr.params
    score = torch.empty(P, dtype=torch.float32, device=dev)
    coords = torch.empty((P, 4), dtype=torch.int32, device=dev)
    if P:
        with torch.cuda.device(dev):
            need = nat.lib.gfx_align_workspace_bytes(P, pr.max_t)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            nat.check(nat.lib.gfx_align(
                q.data_ptr() if len(q) else None, len(q), t.data_ptr() if len(t) else None, len(t),
                pr.pairs_dev.data_ptr(), P, th, go, ge, score.data_ptr(), coords.data_ptr(),
                ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream))
    return score, coords


def _parameters(offset, gap_open, gap_extend):
    vals = []
    for name, v in (("gap_open", gap_open), ("gap_extend", gap_extend), ("offset", offset)):
        if isinstance(v, bool) or not isinstance(v, (int, float, np.floating, np.integer)):
            raise TypeError(f"{name} must be a real number")
        with np.errstate(over="ignore"):
            f = float(np.float32(v))
        if not math.isfinite(f):
            raise ValueError(f"{name} must be finite (as float32)")
        vals.append(f)
    if not (vals[0] > 0 and vals[1] > 0):
        raise ValueError("gap_open and gap_extend must be positive")
    return vals


def _device(device, *tables):
    if device is not None:
        dev = torch.device(device)
    else:
        dev = next((a.device for a in tables if isinstance(a, torch.Tensor) and a.is_cuda),
                   torch.device("cuda"))
    if dev.type != "cuda":
        raise ValueError("device must be a CUDA device: alignment has no CPU path")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def _table(a, what):
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a))
    if not isinstance(a, torch.Tensor):
        raise TypeError(f"{what} must be a NumPy array or a torch tensor")
    if a.dim() != 2 or a.shape[1] != DIM:
        raise ValueError(f"{what} must be [rows, {DIM}], got {tuple(a.shape)}")
    if a.dtype == torch.float32:
        raise ValueError(f"{what} are float32: alignment supports float16 embeddings only "
                         "(cast with .half() / .astype(np.float16))")
    if a.dtype != torch.float16:
        raise ValueError(f"{what} must be float16, got {str(a.dtype).replace('torch.', '')}")
    return a


def _pairs(pairs, q_rows, t_rows):
    if isinstance(pairs, torch.Tensor):
        if pairs.is_floating_point() or pairs.is_complex() or pairs.dtype == torch.bool:
            raise ValueError("pairs must be an integer array")
        p = pairs.detach().cpu().numpy()
    else:
        p = np.asarray(pairs)
        if p.size == 0:
            p = p.reshape(0, 4).astype(np.int64)
        if p.dtype.kind not in "iu":
            raise ValueError("pairs must be an integer array")
    if p.ndim != 2 or p.shape[1] != 4:
        raise ValueError(f"pairs must be [P, 4] (q_start, q_len, t_start, t_len), got {p.shape}")
    p = np.ascontiguousarray(p, dtype=np.int64)
    qs, ql, ts, tl = p.T
    for name, start, length, rows in (("query", qs, ql, q_rows), ("target", ts, tl, t_rows)):
        bad = (length < 0) | (length > MAX_SEGMENT)
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            raise ValueError(f"pair {i}: {name} length {int(length[i])} is outside 0..{MAX_SEGMENT}")
        bad = (start < 0) | (start > rows - length)
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            raise ValueError(f"pair {i}: {name} segment [{int(start[i])}, "
                             f"{int(start[i] + length[i])}) is outside the table of {rows} rows")
    # rows that carry a stripe's bottom row to the next one: multi-stripe pairs only
    multi = ql > 128
    return p, int(tl[multi].max()) if multi.any() else 0


def _all_finite(table: torch.Tensor) -> bool:
    if len(table) == 0:
        return True
    return bool(torch.isfinite(table).all())
