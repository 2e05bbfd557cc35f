"""NumPy oracle of the local alignment contract of `ginfinity_b200.align_pairs`
(include/gfx.h, K8).  Imported by tests and tools only.

For a similarity matrix S [n, m] (query rows i, target columns j):

    s      = S(i,j) - offset
    E(i,j) = max(H(i,j-1) - gap_open, E(i,j-1) - gap_extend)
    F(i,j) = max(H(i-1,j) - gap_open, F(i-1,j) - gap_extend)
    H(i,j) = max(0, H(i-1,j-1) + s, E(i,j), F(i,j))
    H(-1,.) = H(.,-1) = 0,  E(.,-1) = F(-1,.) = -inf

Tie rules: a positive H takes the first of diagonal, E, F that attains it; a
diagonal step from H = 0 starts at (i, j); opening beats extending; the end is
the largest H, then the smallest i, then the smallest j.

The DP runs over anti-diagonals (every cell of one is independent), in the
dtype of S: float32 gives the kernel's arithmetic operation for operation.
"""
from __future__ import annotations

import numpy as np

NONE = (0.0, -1, -1, -1, -1)


def _dp(S, offset, gap_open, gap_extend, anchor=None):
    """H and the packed start (i << 16 | j) of every cell, as [n+1, m+1] arrays
    with the boundary in row and column 0.  With `anchor` = (i0, j0) only
    alignments that begin with a diagonal step at that cell are allowed (no
    zero floor, -inf elsewhere): H(i, j) is then the best such alignment that
    ends at (i, j)."""
    S = np.asarray(S)
    dt = S.dtype.type
    n, m = S.shape
    go, ge, th = dt(gap_open), dt(gap_extend), dt(offset)
    ninf = dt(-np.inf)
    floor = ninf if anchor is not None else dt(0)
    H = np.full((n + 1, m + 1), floor, dtype=S.dtype)
    E = np.full((n + 1, m + 1), ninf, dtype=S.dtype)
    F = np.full((n + 1, m + 1), ninf, dtype=S.dtype)
    sH = np.zeros((n + 1, m + 1), dtype=np.int64)
    sE = np.zeros_like(sH)
    sF = np.zeros_like(sH)
    for d in range(n + m - 1):
        i = np.arange(max(0, d - m + 1), min(n, d + 1))
        j = d - i
        s = S[i, j] - th
        eo, ee = H[i + 1, j] - go, E[i + 1, j] - ge
        En = np.maximum(eo, ee)
        sEn = np.where(eo >= ee, sH[i + 1, j], sE[i + 1, j])
        fo, fe = H[i, j + 1] - go, F[i, j + 1] - ge
        Fn = np.maximum(fo, fe)
        sFn = np.where(fo >= fe, sH[i, j + 1], sF[i, j + 1])
        hd = H[i, j]
        diag = hd + s
        if anchor is not None:
            at = (i == anchor[0]) & (j == anchor[1])
            diag = np.where(at, s, diag)
            Hn = np.maximum(diag, np.maximum(En, Fn))
            here = np.full(i.shape, (anchor[0] << 16) | anchor[1], dtype=np.int64)
            sdiag = np.where(at, here, sH[i, j])
        else:
            Hn = np.maximum(np.maximum(diag, np.maximum(En, Fn)), dt(0))
            sdiag = np.where(hd == 0, (i << 16) | j, sH[i, j])
        sHn = np.where(diag == Hn, sdiag, np.where(En == Hn, sEn, sFn))
        H[i + 1, j + 1], E[i + 1, j + 1], F[i + 1, j + 1] = Hn, En, Fn
        sH[i + 1, j + 1], sE[i + 1, j + 1], sF[i + 1, j + 1] = sHn, sEn, sFn
    return H, sH


def align_fp32(S, offset, gap_open, gap_extend):
    """(score, query_begin, query_end, target_begin, target_end) of the local
    alignment of a given similarity matrix, in float32 (np.float32(S))."""
    return _result(*_dp(np.asarray(S, dtype=np.float32), offset, gap_open, gap_extend))


def align_exact(q, t, offset, gap_open, gap_extend):
    """The same in float64 with exact dot products of the rows q [n, d] and
    t [m, d] (float16 or float32 inputs are exact in float64 products; the sums
    are float64)."""
    S = np.asarray(q, dtype=np.float64) @ np.asarray(t, dtype=np.float64).T
    return _result(*_dp(S, offset, gap_open, gap_extend))


def anchored_score(S, offset, gap_open, gap_extend, begin, end):
    """Best score of an alignment that begins with a diagonal step at cell
    `begin` = (i0, j0) and ends at cell `end` = (i1, j1) (both inclusive), in
    the dtype of S; -inf when there is none."""
    (i0, j0), (i1, j1) = begin, end
    S = np.asarray(S)
    if not (0 <= i0 <= i1 < S.shape[0] and 0 <= j0 <= j1 < S.shape[1]):
        return -np.inf
    sub = S[i0:i1 + 1, j0:j1 + 1]
    H, _ = _dp(sub, offset, gap_open, gap_extend, anchor=(0, 0))
    return float(H[-1, -1])


def _result(H, sH):
    body = H[1:, 1:]
    if body.size == 0:
        return NONE
    best = body.max()
    if not best > 0:
        return NONE
    flat = int(np.flatnonzero(body == best)[0])       # row-major: smallest i, then smallest j
    i, j = divmod(flat, body.shape[1])
    start = int(sH[i + 1, j + 1])
    return (float(best), start >> 16, i + 1, start & 0xFFFF, j + 1)
