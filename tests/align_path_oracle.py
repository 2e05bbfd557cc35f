"""The traceback contract of `ginfinity_b200.align_paths` (include/gfx.h,
gfx_align_trace), restated on the CPU: the sibling of `oracle.align_oracle`
(score and region), which it uses for the end-cell choice.

`dp_codes` is align_oracle's anti-diagonal DP (without the anchored mode) that
also records each cell's traceback code, the 4 bits the trace kernel records:
bits 0-1 where H came from (0 when H = 0, else the first of diagonal, E, F that
attains it), bit 2 E opened (else extended), bit 3 F opened.  `align_fp32_path`
follows the codes back from the end cell; `path_score` rescores a path."""
import numpy as np

from oracle.align_oracle import NONE, _result

CODE_ZERO, CODE_DIAG, CODE_E, CODE_F, CODE_E_OPEN, CODE_F_OPEN = 0, 1, 2, 3, 4, 8
# path ops (gfx.h): query row with target row, query row with a gap, target row with a gap
OP_M, OP_I, OP_D = 0, 1, 2


def dp_codes(S, offset, gap_open, gap_extend):
    """H and the packed start (i << 16 | j) of every cell as [n+1, m+1] arrays
    (boundary in row and column 0, as align_oracle._dp), and the codes [n, m]."""
    S = np.asarray(S)
    dt = S.dtype.type
    n, m = S.shape
    go, ge, th = dt(gap_open), dt(gap_extend), dt(offset)
    ninf = dt(-np.inf)
    H = np.full((n + 1, m + 1), dt(0), dtype=S.dtype)
    E = np.full((n + 1, m + 1), ninf, dtype=S.dtype)
    F = np.full((n + 1, m + 1), ninf, dtype=S.dtype)
    sH = np.zeros((n + 1, m + 1), dtype=np.int64)
    sE = np.zeros_like(sH)
    sF = np.zeros_like(sH)
    codes = np.zeros((n, m), np.uint8)
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
        Hn = np.maximum(np.maximum(diag, np.maximum(En, Fn)), dt(0))
        sdiag = np.where(hd == 0, (i << 16) | j, sH[i, j])
        sHn = np.where(diag == Hn, sdiag, np.where(En == Hn, sEn, sFn))
        src = np.where(Hn == 0, CODE_ZERO, np.where(diag == Hn, CODE_DIAG, np.where(En == Hn, CODE_E, CODE_F)))
        codes[i, j] = src | np.where(eo >= ee, CODE_E_OPEN, 0) | np.where(fo >= fe, CODE_F_OPEN, 0)
        H[i + 1, j + 1], E[i + 1, j + 1], F[i + 1, j + 1] = Hn, En, Fn
        sH[i + 1, j + 1], sE[i + 1, j + 1], sF[i + 1, j + 1] = sHn, sEn, sFn
    return H, sH, codes


def align_fp32_path(S, offset, gap_open, gap_extend):
    """align_oracle.align_fp32's tuple and the aligned path as a uint8 array of
    ops (OP_*), in forward order: the path the tie rules define, followed back
    from the end cell through the recorded codes.  Empty when the score is 0."""
    H, sH, codes = dp_codes(np.asarray(S, dtype=np.float32), offset, gap_open, gap_extend)
    res = _result(H, sH)
    if res == NONE:
        return res, np.zeros(0, np.uint8)
    _, qb, qe, tb, te = res
    i, j, state, rev = qe - 1, te - 1, CODE_DIAG, []
    while True:
        if i < 0 or j < 0:
            start = (i + 1, j + 1)
            break
        c = int(codes[i, j])
        if state == CODE_DIAG:
            src = c & 3
            if src == CODE_ZERO:
                start = (i + 1, j + 1)
                break
            if src == CODE_DIAG:
                rev.append(OP_M)
                i, j = i - 1, j - 1
            else:
                state = src
        elif state == CODE_E:
            rev.append(OP_D)
            state = CODE_DIAG if c & CODE_E_OPEN else CODE_E
            j -= 1
        else:
            rev.append(OP_I)
            state = CODE_DIAG if c & CODE_F_OPEN else CODE_F
            i -= 1
    if start != (qb, tb) or state != CODE_DIAG or rev[-1] != OP_M:
        raise AssertionError(f"traceback ends at {start}, the DP reports a start at {(qb, tb)}")
    return res, np.array(rev[::-1], np.uint8)


def path_score(S, ops, begin, offset, gap_open, gap_extend):
    """The score of the path `ops` (OP_*) that begins at cell `begin` = (i, j),
    in the dtype of S, in the order of the contract: v = 0 + s at the first M,
    then + s per M, - gap_open per gap opened (after M or after the other gap
    kind), - gap_extend per gap extended."""
    S = np.asarray(S)
    dt = S.dtype.type
    go, ge, th = dt(gap_open), dt(gap_extend), dt(offset)
    ops = np.asarray(ops)
    if len(ops) == 0:
        return dt(0)
    if ops[0] != OP_M:
        raise ValueError("a path starts with M")
    i, j = begin
    v = dt(0) + (S[i, j] - th)
    prev = OP_M
    for op in ops[1:]:
        if op == OP_M:
            i, j = i + 1, j + 1
            v = v + (S[i, j] - th)
        else:
            if op == OP_I:
                i += 1
            else:
                j += 1
            v = v - (ge if op == prev else go)
        prev = op
    return v
