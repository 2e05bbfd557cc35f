"""Local alignment of per-nucleotide embeddings (Smith-Waterman, affine gaps)
on the GPU: K8 of libgfx.so (csrc/gfx_align.cu).

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
    P = len(pairs_host)
    score = torch.empty(P, dtype=torch.float32, device=dev)
    coords = torch.empty((P, 4), dtype=torch.int32, device=dev)
    if P:
        if isinstance(pairs, torch.Tensor) and pairs.device == dev:
            pairs_dev = pairs.to(torch.int64).contiguous()
        else:
            pairs_dev = torch.from_numpy(pairs_host).to(dev, non_blocking=True)
        with torch.cuda.device(dev):
            need = nat.lib.gfx_align_workspace_bytes(P, max_t)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            nat.check(nat.lib.gfx_align(
                q.data_ptr() if len(q) else None, len(q), t.data_ptr() if len(t) else None, len(t),
                pairs_dev.data_ptr(), P, th, go, ge, score.data_ptr(), coords.data_ptr(),
                ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream))
    return Alignments(score, *coords.unbind(1))


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
