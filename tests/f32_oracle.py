"""The search contract over float32 rows, restated on the CPU: the sibling of
`oracle.gine_oracle.exact_scores_fp32` / `topk_exact` (which read fp16
inputs) for `EmbeddingIndex` over float32 embeddings.

The score is the sequential fp32 FMA chain over dimensions 0..127 of the
fp32 inputs; for L2 the difference q_i - x_i is rounded to fp32 first.  An
fp32 FMA is emulated with float64: the product of two fp32 values is exact
in float64, the sum is split exactly by TwoSum, and the one case in which
rounding the float64 sum to fp32 differs from rounding the exact sum -- the
float64 sum lands exactly halfway between two fp32 values -- is decided by
the sign of the TwoSum error.  So this is the correctly rounded fp32 FMA."""
import numpy as np


def fma32(a, b, acc):
    """Correctly rounded fp32 fma(a, b, acc), elementwise (float32 arrays)."""
    p = a.astype(np.float64) * b.astype(np.float64)          # exact
    x = acc.astype(np.float64)
    s = x + p
    bv = s - x
    err = (x - (s - bv)) + (p - bv)                            # s + err == x + p exactly
    r = s.astype(np.float32)
    r64 = r.astype(np.float64)
    other = np.where(r64 < s, np.nextafter(r, np.float32(np.inf)),
                     np.nextafter(r, np.float32(-np.inf))).astype(np.float64)
    tie = (err != 0) & (s == (r64 + other) / 2) & (r64 != s)
    up = err > 0                                               # the exact sum lies above s
    fix = np.where((other > r64) == up, other, r64).astype(np.float32)
    return np.where(tie, fix, r)


def exact_scores_f32(queries, rows, metric="cosine"):
    """queries [Q, d], rows [R, d] float32 -> float32 [Q, R] scores."""
    q = np.asarray(queries, np.float32)
    x = np.asarray(rows, np.float32)
    acc = np.zeros((q.shape[0], x.shape[0]), np.float32)
    for d in range(q.shape[1]):
        if metric == "cosine":
            a, b = np.broadcast_to(q[:, d, None], acc.shape), np.broadcast_to(x[None, :, d], acc.shape)
        elif metric == "l2":
            a = b = q[:, d, None] - x[None, :, d]              # fp32 difference
        else:
            raise ValueError(metric)
        acc = fma32(a, b, acc)
    return acc if metric == "cosine" else -acc


def topk_exact_f32(queries, database, k, metric="cosine", index_base=0):
    """Brute force under `exact_scores_f32`, ordered by (score desc, index
    asc); slots beyond the number of rows hold (-inf, -1).  Small inputs."""
    Q, D = queries.shape[0], database.shape[0]
    val = np.full((Q, k), -np.inf, np.float32)
    idx = np.full((Q, k), -1, np.int64)
    if D == 0 or Q == 0:
        return val, idx
    s = exact_scores_f32(queries, database, metric)
    ids = np.arange(D)
    kk = min(k, D)
    for r in range(Q):
        order = np.lexsort((ids, -s[r].astype(np.float64)))[:kk]
        idx[r, :kk], val[r, :kk] = order + index_base, s[r][order]
    return val, idx


def unit_rows32(rng, n, dim=128):
    a = rng.normal(size=(n, dim))
    return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)


def fp16_collisions(rng, base, n):
    """n rows equal to `base` (fp32 values that fp16 represents exactly) plus,
    in its four largest components, perturbations away from zero below half
    an fp16 ulp: distinct in fp32, all equal after rounding to fp16.  The
    perturbation of row j is scaled by a shuffled step, so the fp32 order is
    not the index order."""
    dims = np.argsort(np.abs(base))[-4:]
    rows = np.repeat(base[None].astype(np.float32), n, axis=0)
    step = rng.permutation(n).astype(np.float64) / n            # distinct, shuffled, in [0, 1)
    for d in dims:
        half_ulp = np.spacing(np.float16(abs(base[d]))).astype(np.float64) / 2
        rows[:, d] = (base[d] + np.sign(base[d]) * 0.9 * half_ulp * step).astype(np.float32)
    return rows


def near_tie_rows(rng, q, n):
    """n rows within ~3e-6 (componentwise) of q: their scores against q lie
    far inside the split scan's certificate margin, but are distinct in fp32."""
    return (q[None] + rng.normal(size=(n, q.shape[0])) * 3e-6).astype(np.float32)
