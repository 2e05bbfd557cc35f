"""K8 local alignment on the GPU (align_pairs / gfx_align) against the NumPy
oracle (oracle/align_oracle.py).

Bit-for-bit tests use rows whose components are in {0, +-1/4, +-1/2} with at
most 16 nonzeros: every partial sum of a dot product is a multiple of 1/16
below 4 in magnitude, exact in fp32 in any summation order, so the tensor-core
S is the exact S and the kernel must reproduce align_fp32 exactly."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.align_oracle import align_exact, align_fp32, anchored_score  # noqa: E402

REL = 2.0 ** -14                  # kAlignRel of gfx_align.cu
DYADIC = (0.5, 1.0, 0.25)         # offset, gap_open, gap_extend: exact ties everywhere
ROUNDED = (0.3, 1.1, 0.35)        # the DP rounds: operation order matters
LENGTHS = (1, 31, 32, 33, 127, 128, 129, 256, 257, 1000, 4096)


@pytest.fixture(scope="module")
def ap():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ginfinity_b200.align import align_pairs
    return align_pairs


def sparse_rows(rng, n):
    x = np.zeros((n, 128), np.float16)
    nnz = rng.integers(1, 17, size=n)
    for r in range(n):
        idx = rng.choice(128, size=nnz[r], replace=False)
        x[r, idx] = rng.choice([-0.5, -0.25, 0.25, 0.5], size=nnz[r])
    return x


def mutate(rng, rows, source):
    """A noisy copy of `rows`: some rows replaced from `source`, some deleted,
    some inserted (so alignments carry gaps of both kinds)."""
    out = []
    for r in rows:
        u = rng.random()
        if u < 0.05:
            continue
        out.append(source[rng.integers(len(source))] if u < 0.15 else r)
        if u > 0.95:
            out.extend(source[rng.integers(len(source), size=rng.integers(1, 4))])
    return np.array(out, np.float16).reshape(-1, 128)


def build_problem(rng, shapes, pad=37):
    """Query and target tables holding one segment per pair, separated by unrelated
    rows (they must not leak into an alignment).  Targets embed a mutated copy of
    part of their query, so alignments are long and carry gaps."""
    filler = sparse_rows(rng, 512)
    qs, ts, pairs, qpos, tpos = [], [], [], 0, 0
    for n, m in shapes:
        q = sparse_rows(rng, n)
        core = mutate(rng, q[rng.integers(0, max(1, n // 3)):], filler)[:m]
        t = sparse_rows(rng, m)
        at = rng.integers(0, m - len(core) + 1)
        t[at:at + len(core)] = core
        lead_q, lead_t = rng.integers(0, pad), rng.integers(0, pad)
        qs += [filler[:lead_q], q]
        ts += [filler[:lead_t], t]
        pairs.append((qpos + lead_q, n, tpos + lead_t, m))
        qpos += lead_q + n
        tpos += lead_t + m
    qs.append(filler[:pad])
    ts.append(filler[:pad])
    return np.concatenate(qs), np.concatenate(ts), np.array(pairs, np.int64)


def expected_fp32(Q, T, pairs, params):
    out = []
    for qs, ql, ts, tl in pairs:
        S = Q[qs:qs + ql].astype(np.float32) @ T[ts:ts + tl].astype(np.float32).T
        out.append(align_fp32(S, *params))
    return out


def run(ap, Q, T, pairs, params, **kw):
    r = ap(Q, T, pairs, offset=params[0], gap_open=params[1], gap_extend=params[2], **kw)
    torch.cuda.synchronize()
    score = r.score.cpu().numpy()
    coords = np.stack([c.cpu().numpy() for c in r[1:]], 1)
    return score, coords


def assert_same(score, coords, want):
    for p, (s, qb, qe, tb, te) in enumerate(want):
        got = (float(score[p]), *map(int, coords[p]))
        assert got == (np.float32(s), qb, qe, tb, te), f"pair {p}: {got} != {(s, qb, qe, tb, te)}"


# ---- 1. bit for bit against the fp32 oracle ----------------------------------------
def boundary_shapes():
    small = [L for L in LENGTHS if L <= 257]
    shapes = [(n, m) for n in small for m in small]
    shapes += [(1000, m) for m in (1, 129, 257, 1000)] + [(n, 1000) for n in (1, 33, 257)]
    shapes += [(4096, 33), (33, 4096), (4096, 4096)]
    return shapes


@pytest.mark.parametrize("params", [DYADIC, ROUNDED], ids=["dyadic", "rounded"])
def test_bit_for_bit_on_every_length_boundary(ap, params):
    rng = np.random.default_rng(11)
    Q, T, pairs = build_problem(rng, boundary_shapes())
    score, coords = run(ap, Q, T, pairs, params)
    assert_same(score, coords, expected_fp32(Q, T, pairs, params))
    assert (score > 0).mean() > 0.9


def test_planted_repeats_tie_on_the_first_end(ap):
    """The target holds the same copy of a query region twice: two ends of equal
    score in the same row; the smaller column wins, with its own start."""
    rng = np.random.default_rng(3)
    for n, gap_rows in ((40, 5), (150, 90), (300, 200)):
        q = sparse_rows(rng, n)
        other = sparse_rows(rng, gap_rows)
        t = np.concatenate([other[:3], q, other, q, other[:7]])
        pairs = np.array([[0, n, 0, len(t)]])
        score, coords = run(ap, q, t, pairs, DYADIC)
        want = expected_fp32(q, t, pairs, DYADIC)
        assert_same(score, coords, want)
        assert 3 <= want[0][3] and want[0][4] <= 3 + n       # inside the first copy
    # planted equal starts: the query repeated, aligned to a single copy
    q0 = sparse_rows(rng, 60)
    q = np.concatenate([q0, q0])
    t = np.concatenate([sparse_rows(rng, 10), q0, sparse_rows(rng, 10)])
    pairs = np.array([[0, len(q), 0, len(t)]])
    for params in (DYADIC, ROUNDED):
        score, coords = run(ap, q, t, pairs, params)
        assert_same(score, coords, expected_fp32(q, t, pairs, params))


# ---- 2. random fp16 unit rows against the float64 optimum ------------------------------
def unit_rows(rng, n):
    x = rng.standard_normal((n, 128))
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float16)


def test_random_unit_rows_within_the_stated_bound(ap):
    rng = np.random.default_rng(21)
    Q = unit_rows(rng, 30000)
    T = unit_rows(rng, 60000)
    P = 100_000
    pairs = np.stack([rng.integers(0, len(Q) - 200, P), np.full(P, 200),
                      rng.integers(0, len(T) - 400, P), np.full(P, 400)], 1)
    # plant a noisy copy of part of the query in some targets, so alignments are long
    planted = rng.choice(P, 300, replace=False)
    for p in planted:
        qs, _, ts, _ = pairs[p]
        off = rng.integers(0, 200)
        noise = Q[qs:qs + 200].astype(np.float64) + 0.3 * rng.standard_normal((200, 128)) / np.sqrt(128)
        T[ts + off:ts + off + 200] = (noise / np.linalg.norm(noise, axis=1, keepdims=True)).astype(np.float16)
    params = (0.02, 0.3, 0.05)
    score, coords = run(ap, Q, T, pairs, params)
    checked = np.concatenate([planted[:100], rng.choice(P, 100, replace=False)])
    for p in checked:
        qs, ql, ts, tl = pairs[p]
        q, t = Q[qs:qs + ql], T[ts:ts + tl]
        best = align_exact(q, t, *params)[0]
        mq = np.linalg.norm(q.astype(np.float64), axis=1).max()
        mt = np.linalg.norm(t.astype(np.float64), axis=1).max()
        bound = min(ql, tl) * REL * mq * mt + (ql + tl) * 2.0 ** -24 * max(best, 1.0)
        assert abs(float(score[p]) - best) <= bound, (p, float(score[p]), best, bound)
        qb, qe, tb, te = map(int, coords[p])
        if best > bound:
            S = q.astype(np.float64) @ t.astype(np.float64).T
            region = anchored_score(S, *params, (qb, tb), (qe - 1, te - 1))
            assert region >= best - 2 * bound, (p, region, best)


# ---- 3. edge cases -----------------------------------------------------------------------
def test_edge_cases(ap):
    rng = np.random.default_rng(4)
    Q = sparse_rows(rng, 300)
    T = sparse_rows(rng, 300)
    pairs = np.array([[0, 0, 0, 10], [5, 10, 0, 0], [0, 0, 0, 0], [300, 0, 300, 0], [0, 50, 0, 50]])
    score, coords = run(ap, Q, T, pairs, DYADIC)
    assert (score[:4] == 0).all() and (coords[:4] == -1).all()
    assert_same(score[4:], coords[4:], expected_fp32(Q, T, pairs[4:], DYADIC))
    # offset above every dot product: nothing is positive
    score, coords = run(ap, Q, T, np.array([[0, 300, 0, 300], [10, 129, 20, 1]]), (4.5, 1.0, 1.0))
    assert (score == 0).all() and (coords == -1).all()
    # no pairs
    score, coords = run(ap, Q, T, np.zeros((0, 4), np.int64), DYADIC)
    assert score.shape == (0,) and coords.shape == (0, 4)
    # one table for both sides, pairs that share and overlap rows
    X = torch.from_numpy(sparse_rows(rng, 700)).cuda()
    pairs = np.array([[0, 300, 0, 300], [0, 300, 100, 300], [100, 300, 0, 300], [50, 500, 40, 600],
                      [0, 300, 0, 300]])
    score, coords = run(ap, X, X, torch.from_numpy(pairs).cuda(), ROUNDED)
    Xh = X.cpu().numpy()
    assert_same(score, coords, expected_fp32(Xh, Xh, pairs, ROUNDED))


# ---- 4. determinism ------------------------------------------------------------------------
def test_results_do_not_depend_on_batch_position_or_table_offset(ap):
    rng = np.random.default_rng(8)
    shapes = [(int(a), int(b)) for a, b in rng.integers(1, 700, size=(60, 2))]
    Q, T, pairs = build_problem(rng, shapes)
    base_s, base_c = run(ap, Q, T, pairs, ROUNDED)
    again_s, again_c = run(ap, Q, T, pairs, ROUNDED)
    assert base_s.tobytes() == again_s.tobytes() and (base_c == again_c).all()
    # shuffled, inside a larger batch, with the tables shifted by 1000 rows
    extra_q, extra_t, extra = build_problem(rng, [(int(a), int(b)) for a, b in rng.integers(1, 900, (200, 2))])
    Q2 = np.concatenate([sparse_rows(rng, 1000), Q, extra_q])
    T2 = np.concatenate([sparse_rows(rng, 1000), T, extra_t])
    moved = pairs + np.array([1000, 0, 1000, 0])
    extra = extra + np.array([1000 + len(Q), 0, 1000 + len(T), 0])
    allp = np.concatenate([moved, extra])
    order = rng.permutation(len(allp))
    s2, c2 = run(ap, Q2, T2, allp[order], ROUNDED)
    where = np.argsort(order)[:len(pairs)]
    assert s2[where].tobytes() == base_s.tobytes() and (c2[where] == base_c).all()


# ---- 5. real encoder output --------------------------------------------------------------
def test_encoder_output_aligns_with_itself(ap, golden_shard, parity):
    import ginfinity_b200 as g
    enc = g.Ginfinity.load("cuda:0", model_dir=parity.model_dir)
    ds = g.DeviceShard.from_shard(golden_shard, "cuda:0")
    emb = enc.encode_device_shard(ds)                       # device route: [N, 128] float16
    ptr = ds.node_ptr.cpu().numpy()
    B = len(ptr) - 1
    lens = np.diff(ptr)
    theta, big = 0.5, 1000.0
    self_pairs = np.stack([ptr[:-1], lens, ptr[:-1], lens], 1)
    score, coords = run(ap, emb, emb, torch.from_numpy(self_pairs).cuda(), (theta, big, big))
    E = emb.cpu().numpy()
    for b in range(B):
        L = int(lens[b])
        e = E[ptr[b]:ptr[b + 1]].astype(np.float64)
        want = float(((e * e).sum(1) - theta).sum())
        norm = np.linalg.norm(e, axis=1).max()
        bound = L * REL * norm * norm + 2 * L * 2.0 ** -24 * max(want, 1.0)
        assert tuple(coords[b]) == (0, L, 0, L), (b, coords[b])
        assert abs(float(score[b]) - want) <= bound
    # each record against [other, itself, other] lands on the middle
    rows, pairs, expect = [], [], []
    pos = 0
    for b in range(B):
        o1, o2 = (b + 1) % B, (b + 2) % B
        seg = np.concatenate([E[ptr[o1]:ptr[o1 + 1]], E[ptr[b]:ptr[b + 1]], E[ptr[o2]:ptr[o2 + 1]]])
        rows.append(seg)
        pairs.append((ptr[b], lens[b], pos, len(seg)))
        expect.append((0, lens[b], lens[o1], lens[o1] + lens[b]))
        pos += len(seg)
    T = np.concatenate(rows)
    score, coords = run(ap, E, T, np.array(pairs, np.int64), (theta, big, big))
    for b in range(B):
        assert tuple(coords[b]) == tuple(int(v) for v in expect[b]), (b, coords[b], expect[b])
