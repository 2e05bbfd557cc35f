"""Alignment traceback on the GPU (align_paths / gfx_align_trace) against the
NumPy oracle's path (tests/align_path_oracle.py: align_fp32_path, path_score).

The bit-for-bit tests use test_gpu_align's sparse dyadic rows, whose tensor-core
S is exact, so every path must equal the oracle's byte for byte."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from align_path_oracle import OP_D, OP_I, OP_M, align_fp32_path, path_score  # noqa: E402
from oracle.align_oracle import align_exact  # noqa: E402
from test_gpu_align import (DYADIC, REL, ROUNDED, boundary_shapes, build_problem,  # noqa: E402
                            sparse_rows, unit_rows)


@pytest.fixture(scope="module")
def al():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ginfinity_b200 import align
    return align


def run_paths(al, Q, T, pairs, params, **kw):
    res, paths = al.align_paths(Q, T, pairs, offset=params[0], gap_open=params[1], gap_extend=params[2], **kw)
    torch.cuda.synchronize()
    score = res.score.cpu().numpy()
    coords = np.stack([c.cpu().numpy() for c in res[1:]], 1)
    ops, offs, lens = paths.ops.cpu().numpy(), paths.offsets.cpu().numpy(), paths.lengths.cpu().numpy()
    return score, coords, [ops[o:o + n] for o, n in zip(offs, lens)], paths


def run_pairs(al, Q, T, pairs, params):
    r = al.align_pairs(Q, T, pairs, offset=params[0], gap_open=params[1], gap_extend=params[2])
    torch.cuda.synchronize()
    return r.score.cpu().numpy(), np.stack([c.cpu().numpy() for c in r[1:]], 1)


def trace_direct(al, Q, T, pairs, params):
    """gfx_align_trace on the pairs as given (no boxes): score, coords, paths."""
    nat = al.nat
    dev = torch.device("cuda", torch.cuda.current_device())
    q = torch.from_numpy(Q).to(dev)
    t = torch.from_numpy(T).to(dev)
    P = len(pairs)
    cap = np.maximum(pairs[:, 1] + pairs[:, 3] - 1, 0)
    offs = np.concatenate([[0], np.cumsum(cap)[:-1]]).astype(np.int64)
    code_bytes = int((pairs[:, 1] * ((pairs[:, 3] + 31) // 32) * 16).sum())
    need = nat.lib.gfx_align_trace_workspace_bytes(P, code_bytes)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    pd = torch.from_numpy(pairs.astype(np.int64)).to(dev)
    od = torch.from_numpy(offs).to(dev)
    score = torch.empty(P, dtype=torch.float32, device=dev)
    coords = torch.empty((P, 4), dtype=torch.int32, device=dev)
    ops = torch.empty(max(int(cap.sum()), 1), dtype=torch.uint8, device=dev)
    lens = torch.empty(P, dtype=torch.int32, device=dev)
    nat.check(nat.lib.gfx_align_trace(q.data_ptr(), len(q), t.data_ptr(), len(t), pd.data_ptr(), P,
                                      params[0], params[1], params[2], score.data_ptr(), coords.data_ptr(),
                                      ops.data_ptr(), od.data_ptr(), lens.data_ptr(), ws.data_ptr(), need,
                                      torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ops, lens = ops.cpu().numpy(), lens.cpu().numpy()
    return score.cpu().numpy(), coords.cpu().numpy(), [ops[o:o + n] for o, n in zip(offs, lens)], lens


def check_path(ops, qb, qe, tb, te):
    assert len(ops) and ops[0] == OP_M and ops[-1] == OP_M
    assert (ops == OP_M).sum() + (ops == OP_I).sum() == qe - qb
    assert (ops == OP_M).sum() + (ops == OP_D).sum() == te - tb


def segment_S(Q, T, pair, dtype=np.float32):
    qs, ql, ts, tl = pair
    return Q[qs:qs + ql].astype(dtype) @ T[ts:ts + tl].astype(dtype).T


# ---- 1. byte for byte against the oracle's path, through boxes and on whole pairs ----------
@pytest.mark.parametrize("params", [DYADIC, ROUNDED], ids=["dyadic", "rounded"])
def test_paths_byte_for_byte_on_every_length_boundary(al, params):
    rng = np.random.default_rng(11)
    Q, T, pairs = build_problem(rng, boundary_shapes())
    score, coords, paths, _ = run_paths(al, Q, T, pairs, params)
    ps, pc = run_pairs(al, Q, T, pairs, params)
    assert score.tobytes() == ps.tobytes() and (coords == pc).all()
    d_score, d_coords, d_paths, d_lens = trace_direct(al, Q, T, pairs, params)
    assert d_score.tobytes() == ps.tobytes() and (d_coords == pc).all()
    for p, pair in enumerate(pairs):
        S = segment_S(Q, T, pair)
        want, ops = align_fp32_path(S, *params)
        got = (float(score[p]), *map(int, coords[p]))
        assert got == (np.float32(want[0]), *want[1:]), (p, got, want)
        assert paths[p].tobytes() == ops.tobytes(), (p, tuple(pair), len(paths[p]), len(ops))
        assert d_paths[p].tobytes() == ops.tobytes(), (p, tuple(pair), int(d_lens[p]), len(ops))
        if want[0] > 0:
            v = path_score(S, paths[p], (want[1], want[3]), *params)
            assert v.tobytes() == np.float32(score[p]).tobytes()
    assert (score > 0).mean() > 0.9


# ---- 2. random unit rows ----------------------------------------------------------------------
def test_random_unit_rows_give_valid_paths_within_the_stated_bound(al):
    rng = np.random.default_rng(21)
    Q = unit_rows(rng, 30000)
    T = unit_rows(rng, 60000)
    P = 100_000
    pairs = np.stack([rng.integers(0, len(Q) - 200, P), np.full(P, 200),
                      rng.integers(0, len(T) - 400, P), np.full(P, 400)], 1)
    planted = rng.choice(P, 300, replace=False)
    for p in planted:
        qs, _, ts, _ = pairs[p]
        off = rng.integers(0, 200)
        noise = Q[qs:qs + 200].astype(np.float64) + 0.3 * rng.standard_normal((200, 128)) / np.sqrt(128)
        T[ts + off:ts + off + 200] = (noise / np.linalg.norm(noise, axis=1, keepdims=True)).astype(np.float16)
    params = (0.02, 0.3, 0.05)
    score, coords, paths, _ = run_paths(al, Q, T, pairs, params)      # the box check did not fire
    ps, pc = run_pairs(al, Q, T, pairs, params)
    assert score.tobytes() == ps.tobytes() and (coords == pc).all()
    lens = np.array([len(x) for x in paths])
    assert ((lens > 0) == (score > 0)).all()
    checked = np.concatenate([planted[:100], rng.choice(P, 100, replace=False)])
    for p in checked:
        qs, ql, ts, tl = pairs[p]
        q, t = Q[qs:qs + ql], T[ts:ts + tl]
        best = align_exact(q, t, *params)[0]
        mq = np.linalg.norm(q.astype(np.float64), axis=1).max()
        mt = np.linalg.norm(t.astype(np.float64), axis=1).max()
        bound = min(ql, tl) * REL * mq * mt + (ql + tl) * 2.0 ** -24 * max(best, 1.0)
        if score[p] == 0:
            assert best <= bound
            continue
        qb, qe, tb, te = map(int, coords[p])
        check_path(paths[p], qb, qe, tb, te)
        v = path_score(segment_S(Q, T, pairs[p], np.float64), paths[p], (qb, tb), *params)
        assert abs(v - best) <= 2 * bound, (p, v, best, bound)


# ---- 3. edge cases, determinism, chunks ---------------------------------------------------------
def test_edge_cases(al):
    rng = np.random.default_rng(4)
    Q = sparse_rows(rng, 300)
    T = sparse_rows(rng, 300)
    pairs = np.array([[0, 0, 0, 10], [5, 10, 0, 0], [0, 0, 0, 0], [300, 0, 300, 0], [0, 50, 0, 50]])
    score, coords, paths, obj = run_paths(al, Q, T, pairs, DYADIC)
    assert (score[:4] == 0).all() and all(len(x) == 0 for x in paths[:4])
    assert paths[4].tobytes() == align_fp32_path(segment_S(Q, T, pairs[4]), *DYADIC)[1].tobytes()
    assert obj.cigars()[:4] == [""] * 4
    # all negative
    score, coords, paths, obj = run_paths(al, Q, T, np.array([[0, 300, 0, 300], [10, 129, 20, 1]]),
                                          (4.5, 1.0, 1.0))
    assert (score == 0).all() and all(len(x) == 0 for x in paths) and len(obj.ops) == 0
    # single-cell alignments: one matching row each, everything else far below the offset
    x = np.zeros((3, 128), np.float16)
    x[1, 0] = 1.0
    y = np.zeros((5, 128), np.float16)
    y[3, 0] = 1.0
    score, coords, paths, obj = run_paths(al, x, y, np.array([[0, 3, 0, 5], [1, 1, 3, 1]]), (0.5, 1.0, 1.0))
    assert obj.cigars() == ["1M", "1M"] and tuple(coords[0]) == (1, 2, 3, 4)
    # no pairs
    score, coords, paths, obj = run_paths(al, Q, T, np.zeros((0, 4), np.int64), DYADIC)
    assert score.shape == (0,) and paths == [] and obj.cigars() == []
    # one table for both sides, pairs that share and overlap rows
    X = torch.from_numpy(sparse_rows(rng, 700)).cuda()
    pairs = np.array([[0, 300, 0, 300], [0, 300, 100, 300], [100, 300, 0, 300], [50, 500, 40, 600],
                      [0, 300, 0, 300]])
    score, coords, paths, _ = run_paths(al, X, X, torch.from_numpy(pairs).cuda(), ROUNDED)
    Xh = X.cpu().numpy()
    for p, pair in enumerate(pairs):
        assert paths[p].tobytes() == align_fp32_path(segment_S(Xh, Xh, pair), *ROUNDED)[1].tobytes()


def test_paths_do_not_depend_on_batch_position_table_offset_or_chunks(al, monkeypatch):
    rng = np.random.default_rng(8)
    shapes = [(int(a), int(b)) for a, b in rng.integers(1, 700, size=(60, 2))]
    Q, T, pairs = build_problem(rng, shapes)
    base_s, base_c, base_p, _ = run_paths(al, Q, T, pairs, ROUNDED)
    extra_q, extra_t, extra = build_problem(rng, [(int(a), int(b)) for a, b in rng.integers(1, 900, (200, 2))])
    Q2 = np.concatenate([sparse_rows(rng, 1000), Q, extra_q])
    T2 = np.concatenate([sparse_rows(rng, 1000), T, extra_t])
    moved = pairs + np.array([1000, 0, 1000, 0])
    extra = extra + np.array([1000 + len(Q), 0, 1000 + len(T), 0])
    allp = np.concatenate([moved, extra])
    order = rng.permutation(len(allp))
    s2, c2, p2, _ = run_paths(al, Q2, T2, allp[order], ROUNDED)
    where = np.argsort(order)[:len(pairs)]
    assert s2[where].tobytes() == base_s.tobytes() and (c2[where] == base_c).all()
    assert all(p2[w].tobytes() == b.tobytes() for w, b in zip(where, base_p))
    # a budget of a few boxes per call: many chunks, the same ops
    one_s, one_c, one_p, one = run_paths(al, Q2, T2, allp, ROUNDED)
    monkeypatch.setattr(al, "CODE_BUDGET", 200_000)
    many_s, many_c, many_p, many = run_paths(al, Q2, T2, allp, ROUNDED)
    assert many_s.tobytes() == one_s.tobytes() and (many_c == one_c).all()
    assert (many.offsets.cpu() == one.offsets.cpu()).all() and (many.lengths.cpu() == one.lengths.cpu()).all()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(many_p, one_p))


# ---- 4. real encoder output ------------------------------------------------------------------
def test_encoder_output_paths(al, golden_shard, parity):
    import ginfinity_b200 as g
    enc = g.Ginfinity.load("cuda:0", model_dir=parity.model_dir)
    ds = g.DeviceShard.from_shard(golden_shard, "cuda:0")
    emb = enc.encode_device_shard(ds)
    ptr = ds.node_ptr.cpu().numpy()
    B = len(ptr) - 1
    lens = np.diff(ptr)
    E = emb.cpu().numpy()
    theta, big = 0.5, 1000.0
    # each record inside [other, itself, other]: exactly L M steps
    rows, pairs, pos = [], [], 0
    for b in range(B):
        o1, o2 = (b + 1) % B, (b + 2) % B
        seg = np.concatenate([E[ptr[o1]:ptr[o1 + 1]], E[ptr[b]:ptr[b + 1]], E[ptr[o2]:ptr[o2 + 1]]])
        rows.append(seg)
        pairs.append((ptr[b], lens[b], pos, len(seg)))
        pos += len(seg)
    T = np.concatenate(rows)
    score, coords, paths, obj = run_paths(al, E, T, np.array(pairs, np.int64), (theta, big, big))
    cig = obj.cigars()
    for b in range(B):
        L = int(lens[b])
        assert paths[b].tobytes() == bytes(L) and cig[b] == f"{L}M", (b, cig[b])
    # each record against a copy with one block of rows deleted, moderate gaps
    rng = np.random.default_rng(2)
    params = (0.3, 0.5, 0.1)
    rows, pairs, pos = [], [], 0
    for b in range(B):
        L = int(lens[b])
        cut = int(rng.integers(0, max(1, L - 4)))
        seg = np.delete(E[ptr[b]:ptr[b + 1]], np.arange(cut, min(L, cut + 4)), axis=0)
        rows.append(seg)
        pairs.append((ptr[b], L, pos, len(seg)))
        pos += len(seg)
    T = np.concatenate(rows)
    pairs = np.array(pairs, np.int64)
    score, coords, paths, _ = run_paths(al, E, T, pairs, params)      # the box check did not fire
    for b in range(B):
        if score[b] == 0:
            continue
        qb, qe, tb, te = map(int, coords[b])
        check_path(paths[b], qb, qe, tb, te)
        S = segment_S(E, T, pairs[b], np.float64)
        v = path_score(S, paths[b], (qb, tb), *params)
        q = E[ptr[b]:ptr[b + 1]].astype(np.float64)
        norm = np.linalg.norm(q, axis=1).max()
        bound = min(qe - qb, te - tb) * REL * norm * norm + (qe - qb + te - tb) * 2.0 ** -24 * max(v, 1.0)
        assert abs(v - float(score[b])) <= bound, (b, v, float(score[b]), bound)
