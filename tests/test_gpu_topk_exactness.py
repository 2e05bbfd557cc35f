"""K5 exactness where the tensor-core candidate choice and the exact score
disagree.  The scan keeps kc = min((k + 7) & ~3, 28) candidates per database
segment, ranked by the tensor-core score; the returned scores are the
sequential fp32 FMA chain of `oracle.gine_oracle.exact_scores_fp32`.  Every
case here is built so that the two orders differ by more than the kc - k
spare candidates, and every search result must equal `O.topk_exact` to the
bit: indices and float32 scores.

Constructions (CPU checks at the top keep them honest):

1. cosine, order-dependent rounding: with q[i0] = q[i1] = 1 and
   q[s1] = q[s2] = 2^-12, row A (x[i0] = 1, x[s1] = x[s2] = 2^-12) and row B
   (x[s1] = x[s2] = 2^-12, x[i1] = 1), i0 < s1 < s2 < i1, have the same real
   dot product 1 + 2^-23.  The sequential chain absorbs A's two 2^-24 terms
   into the leading 1 (ties to even) and scores A at 1.0, while B's small
   terms add up first and B scores 1 + 2^-23.  A summation in another order
   ranks A at or above B, and ties keep the lower index, so kc copies of A in
   front of k rows B push every B out of the candidate list.
2. L2, cancellation: the scan ranks by 2 q.d - |d|^2 in fp32, one ulp of
   which is ~N^2 * 2^-23 for rows of norm N; rows one to three fp16 ulps away
   from the query differ in -|q-d|^2 by far less, so the scan cannot order
   them, while the sequential chain over q - d does.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import gine_oracle as O  # noqa: E402

DIM = 128
SMALL = np.float16(2.0 ** -12)
# (i0, s1, s2, i1): A's leading 1 at i0, the small terms at s1 < s2, B's 1 at i1.
# The first two lie inside one 16-wide K block of the MMA; the last two put the
# terms of a row in K blocks 0 and 7.
LAYOUTS = [(0, 1, 2, 3), (16, 20, 21, 31), (0, 1, 2, 127), (3, 8, 120, 124)]
KS = [1, 4, 5, 8, 20, 21, 24]          # kc - k = 7, 4, 7, 4, 4, 7 and 4 (kc capped at 28)
SAMPLE_ROWS = 128 * 128                # rows of the threshold-seeding pre-pass


def kc_of(k):
    """Candidates the scan keeps per segment (make_plan in csrc/gfx_topk.cu)."""
    return min((k + 7) & ~3, 28)


def segment_rows(Q, D):
    """Rows per database segment of the scan (make_plan in csrc/gfx_topk.cu)."""
    tiles_q, tiles_db = -(-Q // 256), -(-D // 128)
    segs = -(-8 * 148 // tiles_q) if tiles_q < 8 * 148 else 1
    segs = min(segs, max(tiles_db // 16, 1))
    return -(-tiles_db // segs) * 128


def unit_rows(rng, n):
    a = rng.normal(size=(n, DIM)).astype(np.float32)
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    return a.astype(np.float16)


def cosine_pair(layout):
    """(query, row A, row B) of construction 1."""
    i0, s1, s2, i1 = layout
    q, a, b = (np.zeros(DIM, np.float16) for _ in range(3))
    q[[i0, i1]] = 1
    q[[s1, s2]] = SMALL
    a[i0] = 1
    a[[s1, s2]] = SMALL
    b[[s1, s2]] = SMALL
    b[i1] = 1
    return q, a, b


def plant(db, start, first, second, n_first, n_second):
    db[start:start + n_first] = first
    db[start + n_first:start + n_first + n_second] = second


def l2_group(rng, norm, n=64):
    """Construction 2: a row of the given norm (the query), n - 1 rows one to
    three fp16 ulps away from it in one component, the row itself last."""
    base = (unit_rows(rng, 1)[0].astype(np.float32) * norm).astype(np.float16)
    rows = np.repeat(base[None], n, axis=0)
    for r in range(n - 1):
        d = rng.integers(DIM)
        step = np.float16(np.inf) if rng.random() < 0.5 else np.float16(-np.inf)
        for _ in range(rng.integers(1, 4)):
            rows[r, d] = np.nextafter(rows[r, d], step)
    return base, rows


def scan_l2_scores(q, rows):
    """The scan's L2 ranking value 2 q.d - |d|^2 in fp32: q.d and |d|^2 as
    sequential fp32 chains, combined by one fma (fmaf(2, q.d, -|d|^2))."""
    qd = O.exact_scores_fp32(q[None], rows, "cosine")[0].astype(np.float64)
    d2 = np.array([O.exact_scores_fp32(r[None], r[None], "cosine")[0, 0] for r in rows], np.float64)
    return (2.0 * qd - d2).astype(np.float32)


# ---------------- CPU checks of the constructions ------------------------------------------


@pytest.mark.parametrize("layout", LAYOUTS)
def test_cosine_construction_ranks_b_above_a_with_equal_real_dots(layout):
    q, a, b = cosine_pair(layout)
    rows = np.stack([a, b])
    exact = O.exact_scores_fp32(q[None], rows, "cosine")[0]
    real = rows.astype(np.float64) @ q.astype(np.float64)
    assert real[0] == real[1] == 1 + 2.0 ** -23
    assert exact[0] == np.float32(1.0) and exact[1] == np.float32(1 + 2.0 ** -23)
    val, idx = O.topk_exact(q[None], rows, 2, "cosine")
    assert list(idx[0]) == [1, 0]


@pytest.mark.parametrize("norm", [30, 100, 1000])
def test_l2_construction_defeats_the_scan_ranking(norm):
    rng = np.random.default_rng(norm)
    q, rows = l2_group(rng, norm)
    ids = np.arange(len(rows))
    exact = O.exact_scores_fp32(q[None], rows, "l2")[0]
    diff = rows.astype(np.float64) - q.astype(np.float64)
    real = -(diff * diff).sum(axis=1)
    order_exact = np.lexsort((ids, -exact.astype(np.float64)))
    order_real = np.lexsort((ids, -real))
    np.testing.assert_array_equal(order_exact, order_real)
    assert order_exact[0] == len(rows) - 1 and exact[-1] == 0       # the row itself first
    scan = scan_l2_scores(q, rows)
    assert len(np.unique(scan)) <= 8                                # 64 rows, a handful of values
    assert scan[-1] <= scan[:-1].max()                              # the row itself is not ahead


@pytest.mark.parametrize("Q,D,k", [(1, 40_000, 1), (300, 20_000, 24), (2048, 1_000_000, 10),
                                   (100_000, 12_500_000, 10)])
def test_workspace_holds_every_region(Q, D, k):
    """gfx_topk's workspace: a 256-byte header (fallback count, largest squared
    norm), the flagged-query list, candidate scores and indices of every
    segment, the squared row norms and, for >= 131,072 rows, the seed lists --
    none of them overlapping."""
    try:
        from ginfinity_b200 import _native as nat
    except ImportError:
        pytest.skip("libgfx.so is not built")
    tiles_q, tiles_db = -(-Q // 256), -(-D // 128)
    segs = -(-tiles_db * 128 // segment_rows(Q, D))
    up = lambda v: -(-v // 256) * 256  # noqa: E731
    cand = segs * tiles_q * 256 * kc_of(k)
    need = 256 + up(4 * Q) + 2 * up(4 * cand) + up(4 * tiles_db * 128)
    if tiles_db >= 8 * 128:
        need += 2 * up(4 * tiles_q * 256 * kc_of(k))
    assert nat.lib.gfx_topk_workspace_bytes(Q, D, k) == need


# ---------------- GPU cases ----------------------------------------------------------------


@pytest.fixture(scope="module")
def search():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from ginfinity_b200 import search as S
    return S


def run(search, q, db, k, metric):
    """(scores, index, fallback count) of one search on cuda:0."""
    index = search.EmbeddingIndex(db, device="cuda:0")
    s, i = index.search(q, k, metric)
    torch.cuda.synchronize()
    return s.cpu().numpy(), i.cpu().numpy(), index


def assert_exact(got_s, got_i, want_s, want_i):
    np.testing.assert_array_equal(got_i, want_i)
    np.testing.assert_array_equal(got_s, want_s)


def cosine_database(seed, D, k, layout, start, b_first=False):
    rng = np.random.default_rng(seed)
    db = unit_rows(rng, D)
    q, a, b = cosine_pair(layout)
    if b_first:
        plant(db, start, b, a, k, kc_of(k))
    else:
        plant(db, start, a, b, kc_of(k), k)
    return q, db


@pytest.mark.gpu
@pytest.mark.parametrize("Q", [1, 300])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("k", KS)
def test_planted_cosine_near_ties(search, k, layout, Q):
    """kc copies of A, then k rows B, inside the fourth of several segments."""
    D = 40_000
    seg = segment_rows(Q, D)
    assert D // seg >= 4
    q, db = cosine_database(100 + k, D, k, layout, 3 * seg + 40)
    want_s, want_i = O.topk_exact(q[None], db, k, "cosine")
    assert np.all(want_s == np.float32(1 + 2.0 ** -23))             # the k rows B
    got_s, got_i, index = run(search, np.repeat(q[None], Q, axis=0), db, k, "cosine")
    assert_exact(got_s, got_i, np.repeat(want_s, Q, 0), np.repeat(want_i, Q, 0))
    assert index.last_fallbacks() == Q


@pytest.mark.gpu
@pytest.mark.parametrize("Q", [1, 300])
@pytest.mark.parametrize("k", KS)
def test_planted_cosine_mirror_order(search, k, Q):
    """The rows B before the copies of A: the scan keeps them either way."""
    D = 40_000
    q, db = cosine_database(200 + k, D, k, LAYOUTS[1], 2 * segment_rows(Q, D) + 7, b_first=True)
    want_s, want_i = O.topk_exact(q[None], db, k, "cosine")
    got_s, got_i, _ = run(search, np.repeat(q[None], Q, axis=0), db, k, "cosine")
    assert_exact(got_s, got_i, np.repeat(want_s, Q, 0), np.repeat(want_i, Q, 0))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 10, 24])
@pytest.mark.parametrize("norm", [30, 100, 1000])
def test_planted_l2_cancellation(search, norm, k):
    """Eight groups of construction 2, one per segment, each group's row as a
    query: its first result is the row itself at score 0."""
    rng = np.random.default_rng(norm * 31 + k)
    D, Q = 20_000, 8
    db = (unit_rows(rng, D).astype(np.float32) * norm).astype(np.float16)
    seg = segment_rows(Q, D)
    assert D // seg >= Q
    q = np.empty((Q, DIM), np.float16)
    for g in range(Q):
        q[g], rows = l2_group(rng, norm)
        db[g * seg + 11:g * seg + 11 + len(rows)] = rows
    want_s, want_i = O.topk_exact(q, db, k, "l2")
    assert np.all(want_i[:, 0] == np.arange(Q) * seg + 11 + 63) and np.all(want_s[:, 0] == 0)
    got_s, got_i, index = run(search, q, db, k, "l2")
    assert_exact(got_s, got_i, want_s, want_i)
    assert index.last_fallbacks() == Q


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 24])
@pytest.mark.parametrize("where", ["a_in_sample", "b_in_sample", "segment_boundary"])
def test_planted_groups_across_the_seeding_sample_and_segments(search, where, k):
    """Databases of >= 131,072 rows take the threshold-seeding pre-pass over
    the first 16,384 rows.  The copies of A and the rows B lie on different
    sides of that sample, or on both sides of a segment boundary."""
    D, Q = 140_000, 4
    rng = np.random.default_rng(300 + k)
    db = unit_rows(rng, D)
    q, a, b = cosine_pair(LAYOUTS[3])
    kc = kc_of(k)
    seg = segment_rows(Q, D)
    if where == "a_in_sample":
        db[1000:1000 + kc], db[100_000:100_000 + k] = a, b
    elif where == "b_in_sample":
        db[2000:2000 + k], db[90_000:90_000 + kc] = b, a
    else:
        edge = 20 * seg
        assert edge > SAMPLE_ROWS
        db[edge - kc:edge], db[edge:edge + k] = a, b
    want_s, want_i = O.topk_exact(q[None], db, k, "cosine")
    assert np.all(want_s == np.float32(1 + 2.0 ** -23))
    got_s, got_i, _ = run(search, np.repeat(q[None], Q, axis=0), db, k, "cosine")
    assert_exact(got_s, got_i, np.repeat(want_s, Q, 0), np.repeat(want_i, Q, 0))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 24])
@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_near_tie_stress_without_a_planted_winner(search, metric, k):
    """Per query ~200 rows one fp16 ulp away from the query in components where
    the query is at most 2^-8, shuffled and scattered over the database."""
    rng = np.random.default_rng(400 + k + (metric == "l2"))
    D, Q, n = 50_000, 16, 200
    db = unit_rows(rng, D)
    q = unit_rows(rng, Q)
    small = np.zeros((Q, DIM), bool)
    for r in range(Q):                      # 16 components of every query at most 2^-8
        dims = rng.choice(DIM, 16, replace=False)
        q[r, dims] = (rng.uniform(-1, 1, 16) * 2.0 ** -8).astype(np.float16)
        small[r, dims] = True
    assert np.all(np.abs(q[small].astype(np.float32)) <= 2.0 ** -8)
    planted = []
    for r in range(Q):
        dims = np.flatnonzero(small[r])
        for _ in range(n):
            row = q[r].copy()
            for d in rng.choice(dims, rng.integers(1, 4), replace=False):
                row[d] = np.nextafter(row[d], np.float16(np.inf if rng.random() < 0.5 else -np.inf))
            planted.append(row)
    pos = rng.choice(D, len(planted), replace=False)
    db[pos] = np.stack(planted)[rng.permutation(len(planted))]
    want_s, want_i = O.topk_exact(q, db, k, metric)
    got_s, got_i, _ = run(search, q, db, k, metric)
    assert_exact(got_s, got_i, want_s, want_i)


@pytest.mark.gpu
def test_random_unit_data_stays_on_the_fast_path(search):
    """Q = 2048 x D = 1e6 random unit vectors: no query needs the exact fallback,
    and a subset of 16 queries equals the oracle.  The oracle runs on the rows
    whose float64 score is within 1e-4 of the 10th best: the fp32 chain is within
    128 * 2^-24 * sum|q_i x_i| <= 7.7e-6 of the float64 score for unit vectors,
    so no row outside that set can reach the top 10."""
    rng = np.random.default_rng(500)
    D, Q, k = 1_000_000, 2048, 10
    db, q = unit_rows(rng, D), unit_rows(rng, Q)
    got_s, got_i, index = run(search, q, db, k, "cosine")
    assert index.last_fallbacks() == 0
    sub = rng.choice(Q, 16, replace=False)
    f64 = q[sub].astype(np.float64) @ db.astype(np.float64).T
    for r, f in zip(sub, f64):
        keep = np.flatnonzero(f >= np.sort(f)[-k] - 1e-4)
        want_s, want_i = O.topk_exact(q[r:r + 1], db[keep], k, "cosine")
        assert_exact(got_s[r], got_i[r], want_s[0], keep[want_i[0]])
