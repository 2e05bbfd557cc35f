"""Search over float32 embeddings (EmbeddingIndex of float32 rows, gfx_topk_f32)
against the fp32-row oracle (tests/f32_oracle.py): indices bit for bit and
float32 scores equal, for random cases, rows that only fp32 can order,
near-ties below the split scan's margin, the seeding pre-pass, shards, an
out-of-fp16-range query, argument checks, and the full_precision encoder's
HBM output searched in place."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from f32_oracle import fp16_collisions, near_tie_rows, topk_exact_f32, unit_rows32  # noqa: E402
from oracle import gine_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def search():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from ginfinity_b200 import search as S
    return S


def unit(seed, n, scale=None):
    rng = np.random.default_rng(seed)
    a = unit_rows32(rng, n)
    if scale is not None:
        a *= rng.uniform(*scale, size=(n, 1)).astype(np.float32)
    return a


def run(search, q, db, k, metric, index_base=0):
    index = search.EmbeddingIndex(db, device="cuda:0", index_base=index_base)
    s, i = index.search(q, k, metric)
    torch.cuda.synchronize()
    return s.cpu().numpy(), i.cpu().numpy(), index


def assert_exact(got_s, got_i, want_s, want_i):
    np.testing.assert_array_equal(got_i, want_i)
    np.testing.assert_array_equal(got_s, want_s)


@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("Q,D,k", [(300, 5000, 10), (1, 129, 1), (257, 4096, 24), (64, 127, 5)])
def test_f32_topk_matches_the_exact_oracle(search, metric, Q, D, k):
    q = unit(1, Q)
    db = unit(2, D, scale=(0.5, 1.5) if metric == "l2" else None)
    got_s, got_i, index = run(search, q, db, k, metric)
    assert index.dtype == torch.float32 and got_s.dtype == np.float32 and got_i.dtype == np.int64
    assert_exact(got_s, got_i, *topk_exact_f32(q, db, k, metric))


def test_f32_many_segments_and_query_tiles(search):
    db = unit(9, 40_000)
    for Q in (7, 700):
        q = unit(10 + Q, Q)
        got_s, got_i, _ = run(search, q, db, 10, "cosine", index_base=123)
        sub = np.arange(0, Q, max(1, Q // 40))
        want_s, want_i = topk_exact_f32(q[sub], db, 10, "cosine", index_base=123)
        assert_exact(got_s[sub], got_i[sub], want_s, want_i)


def test_f32_short_and_empty_databases_pad_with_minus_inf(search):
    q, db = unit(7, 33), unit(8, 5)
    s, i, _ = run(search, q, db, 8, "cosine", index_base=1000)
    assert_exact(s, i, *topk_exact_f32(q, db, 8, "cosine", index_base=1000))
    assert np.all(i[:, 5:] == -1) and np.all(np.isneginf(s[:, 5:]))
    s, i, _ = run(search, q, db[:0], 3, "l2")
    assert np.all(i == -1) and np.all(np.isneginf(s))
    s, i, _ = run(search, q[:0], db, 3, "cosine")
    assert s.shape == (0, 3) and i.shape == (0, 3)


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_rows_equal_in_fp16_are_ordered_by_an_fp32_index(search, metric):
    """30 rows that round to one fp16 row, scattered over a database: the fp32
    index returns them in the oracle's fp32 order, which is not index order; the
    same data as fp16 ties, and an fp16 index returns them in index order."""
    rng = np.random.default_rng(30)
    D, k = 20_000, 24
    db = unit_rows32(rng, D)
    base = unit_rows32(rng, 1)[0].astype(np.float16).astype(np.float32)
    pos = np.sort(rng.choice(D, 30, replace=False))
    db[pos] = fp16_collisions(rng, base, 30)
    q = np.stack([base, unit_rows32(rng, 1)[0]])
    got_s, got_i, _ = run(search, q, db, k, metric)
    want_s, want_i = topk_exact_f32(q, db, k, metric)
    assert_exact(got_s, got_i, want_s, want_i)
    assert set(got_i[0]) <= set(pos) and not np.all(np.diff(got_i[0]) > 0)   # fp32 order, not index order
    s16, i16, _ = run(search, q.astype(np.float16), db.astype(np.float16), k, metric)
    np.testing.assert_array_equal(i16[0], pos[:k])                           # ties in index order
    assert np.all(s16[0] == s16[0, 0])


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_near_ties_below_the_split_margin_take_the_fallback(search, metric):
    """40 rows within 3e-6 of each query inside one segment: the scan keeps kc of
    them and cannot certify the order, so the query is rescored exactly."""
    rng = np.random.default_rng(40)
    D, Q, k = 40_000, 3, 10
    db = unit_rows32(rng, D)
    q = unit_rows32(rng, Q)
    for r in range(Q):
        start = 5_000 + r * 10_000
        db[start:start + 40] = near_tie_rows(rng, q[r], 40)
    got_s, got_i, index = run(search, q, db, k, metric)
    assert_exact(got_s, got_i, *topk_exact_f32(q, db, k, metric))
    assert index.last_fallbacks() > 0


def test_f32_random_unit_data_stays_on_the_fast_path(search):
    """Q = 2048 x D = 1e6 random fp32 unit vectors: no query needs the fallback;
    16 queries equal the oracle over the rows within 1e-4 of their 10th best
    float64 score (the fp32 chain is within 7.7e-6 of it for unit vectors)."""
    rng = np.random.default_rng(500)
    D, Q, k = 1_000_000, 2048, 10
    db, q = unit_rows32(rng, D), unit_rows32(rng, Q)
    got_s, got_i, index = run(search, q, db, k, "cosine")
    assert index.last_fallbacks() == 0
    sub = rng.choice(Q, 16, replace=False)
    f64 = q[sub].astype(np.float64) @ db.astype(np.float64).T
    for r, f in zip(sub, f64):
        keep = np.flatnonzero(f >= np.sort(f)[-k] - 1e-4)
        want_s, want_i = topk_exact_f32(q[r:r + 1], db[keep], k, "cosine")
        assert_exact(got_s[r], got_i[r], want_s[0], keep[want_i[0]])


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_f32_seeded_scan_on_a_large_database_with_ties(search, metric):
    """>= 131,072 rows take the threshold-seeding pre-pass over the first 16,384
    rows; the best rows are duplicated inside and outside that sample."""
    rng = np.random.default_rng(15)
    D, Q, k = 140_000, 40, 10
    db = unit(16, D, scale=(0.7, 1.3) if metric == "l2" else None)
    q = unit(17, Q)
    hot = db[rng.integers(0, 16_384, 6)]
    for pos in (20_000, 77_777, 139_990):
        db[pos:pos + 6] = hot
    q[:6] = hot
    got_s, got_i, _ = run(search, q, db, k, metric)
    assert_exact(got_s, got_i, *topk_exact_f32(q, db, k, metric))
    assert np.all(got_s[:6, 0] == got_s[:6, 3]) and np.all(np.diff(got_i[:6, :4], axis=1) > 0)


def test_f32_sharded_results_merge_to_the_global_answer(search):
    q, db = unit(11, 150), unit(12, 9000)
    k, world = 10, 3
    parts = [search.EmbeddingIndex.shard(db, rank=r, world_size=world, device="cuda:0").search(q, k)
             for r in range(world)]
    got_s, got_i = search.merge_lists(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    torch.cuda.synchronize()
    assert_exact(got_s.cpu().numpy(), got_i.cpu().numpy(), *topk_exact_f32(q, db, k, "cosine"))


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_query_beyond_the_fp16_range_takes_the_fallback(search, metric):
    q, db = unit(20, 3), unit(21, 30_000)
    q[1, 17] = 1e5                      # its fp16 hi part would be inf
    got_s, got_i, index = run(search, q, db, 5, metric)
    assert_exact(got_s, got_i, *topk_exact_f32(q, db, 5, metric))
    assert index.last_fallbacks() == 1


def test_f32_argument_checks(search):
    db, q = unit(13, 10), unit(14, 2)
    index = search.EmbeddingIndex(db, device="cuda:0")
    assert index.dtype == torch.float32
    with pytest.raises(ValueError, match="float32"):
        index.search(q.astype(np.float16), 3)
    with pytest.raises(ValueError, match="float32"):
        index.search(q.astype(np.float64), 3)
    index16 = search.EmbeddingIndex(db.astype(np.float16), device="cuda:0")
    assert index16.dtype == torch.float16
    with pytest.raises(ValueError, match="float16"):
        index16.search(q, 3)
    with pytest.raises(ValueError, match="float16 or float32"):
        search.EmbeddingIndex(db.astype(np.float64), device="cuda:0")
    big = db.copy()
    big[4, 9] = -70_000.0
    with pytest.raises(ValueError, match="65504"):
        search.EmbeddingIndex(big, device="cuda:0")
    big[4, 9] = 65504.0                 # the largest fp16 value is accepted
    search.EmbeddingIndex(big, device="cuda:0")


def test_full_precision_encoder_output_searched_in_hbm(search, synthetic_state):
    """encode_device_shard(out_dtype=GFX_F32) -> EmbeddingIndex without a host
    copy: every nucleotide's best hit is itself (or an identical row before it),
    and the top 3 equal the oracle."""
    import ginfinity_b200 as g
    from ginfinity_b200 import _native as nat
    from ginfinity_b200.device_builder import build_device_shard
    from helpers import random_records
    enc = g.Ginfinity.from_state(synthetic_state, device="cuda:0", full_precision=True)
    ds = build_device_shard(random_records(21, 30), "cuda:0")
    emb = enc.encode_device_shard(ds, out_dtype=nat.GFX_F32)
    assert emb.dtype == torch.float32 and emb.is_cuda
    index = search.EmbeddingIndex(emb, device="cuda:0")
    assert index.database.data_ptr() == emb.data_ptr()
    s, i = index.search(emb[:500], 3, "cosine")
    torch.cuda.synchronize()
    host = emb.cpu().numpy()
    got_s, got_i = s.cpu().numpy(), i.cpu().numpy()
    want_s, want_i = topk_exact_f32(host[:500], host, 3, "cosine")
    assert_exact(got_s, got_i, want_s, want_i)
    me = np.arange(500)
    assert np.all((got_i[:, 0] == me) | np.all(host[got_i[:, 0]] == host[me], axis=1))
    assert np.all(np.abs(got_s[:, 0] - 1.0) < 1e-5)
    # the same embeddings through the fp16 oracle would not be the contract: scores differ
    assert not np.array_equal(got_s, O.topk_exact(host[:500].astype(np.float16),
                                                  host.astype(np.float16), 3, "cosine")[0])
