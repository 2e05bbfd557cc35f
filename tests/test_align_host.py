"""Local alignment (align_pairs / gfx_align) without a GPU: the NumPy oracle
against brute force and hand-built ties, argument errors of the C ABI, and the
Python layer's validation, which runs before any device work."""
import math
import shutil

import numpy as np
import pytest

from oracle.align_oracle import align_exact, align_fp32, anchored_score


def gap(L, go, ge):
    return go + (L - 1) * ge


def brute_force(S, th, go, ge):
    """Best score over every chain of matched cells (strictly increasing i and j);
    between two matches a skip of di rows and dj columns pays one gap per skipped
    dimension."""
    n, m = S.shape
    best = 0.0
    cells = [(i, j) for i in range(n) for j in range(m)]

    def extend(i, j, score):
        nonlocal best
        best = max(best, score)
        for i2 in range(i + 1, n):
            for j2 in range(j + 1, m):
                di, dj = i2 - i - 1, j2 - j - 1
                cost = (gap(di, go, ge) if di else 0.0) + (gap(dj, go, ge) if dj else 0.0)
                extend(i2, j2, score - cost + (S[i2, j2] - th))

    for i, j in cells:
        extend(i, j, S[i, j] - th)
    return best


def dyadic(rng, shape, lo=-4, hi=5):
    return rng.integers(lo, hi, size=shape).astype(np.float32) / 4


@pytest.mark.parametrize("seed", range(40))
def test_fp32_oracle_matches_brute_force_on_small_dyadic_inputs(seed):
    rng = np.random.default_rng(seed)
    n, m = rng.integers(1, 5, size=2)
    S = dyadic(rng, (n, m))
    th, go, ge = 0.25 * rng.integers(0, 3), 0.25 * rng.integers(1, 5), 0.25 * rng.integers(1, 3)
    score, qb, qe, tb, te = align_fp32(S, th, go, ge)
    assert score == brute_force(S.astype(np.float64), th, go, ge)
    if score > 0:
        # the returned region holds an alignment of that score
        assert anchored_score(S, th, go, ge, (qb, tb), (qe - 1, te - 1)) == score
    else:
        assert (qb, qe, tb, te) == (-1, -1, -1, -1)


def test_two_equal_ends_take_the_smaller_row_then_column():
    S = np.zeros((3, 3), np.float32)
    S[0, 2] = S[2, 0] = 1.0
    assert align_fp32(S, 0.0, 1.0, 1.0) == (1.0, 0, 1, 2, 3)
    S = np.zeros((2, 3), np.float32)
    S[1, 0] = S[1, 2] = 1.0
    assert align_fp32(S, 0.0, 1.0, 1.0) == (1.0, 1, 2, 0, 1)


def test_diagonal_wins_over_equal_gaps():
    # H(1,1) can come from the diagonal (1 + 1 - 1 = 1) or from E / F opened at 2 - 1 = 1
    S = np.array([[2.0, 1.0], [1.0, -1.0]], np.float32)
    score, qb, qe, tb, te = align_fp32(S, 0.0, 1.0, 1.0)
    assert score == 2.0 and (qb, qe, tb, te) == (0, 1, 0, 1)
    H_end = anchored_score(S, 0.0, 1.0, 1.0, (0, 0), (1, 1))
    assert H_end == 1.0


def test_e_wins_over_equal_f_and_diagonal_start_rule():
    # cell (1,1): diagonal 0 + 0.5 (new start at (1,1)), E from (1,0), F from (0,1)
    S = np.array([[0.0, 2.0, 0.0], [2.0, 0.5, 0.0]], np.float32)
    # E(1,1) = H(1,0) - 1.5 = 0.5 ; F(1,1) = H(0,1) - 1.5 = 0.5 ; diagonal 0.5: the diagonal wins
    from oracle.align_oracle import _dp
    H, sH = _dp(S, 0.0, 1.5, 1.0)
    assert H[2, 2] == 0.5 and sH[2, 2] == (1 << 16) | 1
    # without the diagonal (S(1,1) very negative) E and F tie; E (the left one) wins
    S[1, 1] = -8.0
    H, sH = _dp(S, 0.0, 1.5, 1.0)
    assert H[2, 2] == 0.5 and sH[2, 2] == (1 << 16) | 0


def test_opening_wins_over_extending():
    # row 0: H(0,0) = 3; H(0,1) = 2 starts anew at (0,1) (diagonal from the boundary beats
    # E(0,1) = 3 - 1 = 2 by the diagonal-first rule); at (0,2) opening from H(0,1) and
    # extending E(0,1) both give 1: the gap is taken as opened at (0,1)
    from oracle.align_oracle import _dp
    S = np.array([[3.0, 2.0, -9.0, 9.0]], np.float32)
    H, sH = _dp(S, 0.0, 1.0, 1.0)
    assert H[1, 2] == 2.0 and sH[1, 2] == (0 << 16) | 1
    assert H[1, 3] == 1.0 and sH[1, 3] == (0 << 16) | 1


def test_exact_oracle_agrees_with_fp32_on_dyadic_inputs():
    rng = np.random.default_rng(5)
    for _ in range(10):
        n, m = rng.integers(1, 30, size=2)
        q = np.zeros((n, 128), np.float16)
        t = np.zeros((m, 128), np.float16)
        for a in (q, t):
            for r in a:
                idx = rng.choice(128, size=8, replace=False)
                r[idx] = rng.choice([-0.5, -0.25, 0.25, 0.5], size=8)
        S = q.astype(np.float32) @ t.astype(np.float32).T
        assert align_exact(q, t, 0.125, 0.5, 0.25) == align_fp32(S, 0.125, 0.5, 0.25)


def test_empty_and_all_negative_give_no_alignment():
    assert align_fp32(np.zeros((0, 5), np.float32), 0.0, 1.0, 1.0) == (0.0, -1, -1, -1, -1)
    assert align_fp32(np.full((3, 3), 0.5, np.float32), 1.0, 1.0, 1.0) == (0.0, -1, -1, -1, -1)


# ---------------------------------------------------------------- C ABI and Python layer

@pytest.fixture(scope="module")
def nat():
    from ginfinity_b200 import build_native
    if not build_native.LIB.is_file() and shutil.which(build_native.NVCC) is None:
        pytest.skip("libgfx.so is not built and nvcc is not installed here")
    if shutil.which(build_native.NVCC) is not None:
        build_native.build()
    from ginfinity_b200 import _native
    return _native


def test_gfx_align_argument_errors_surface_through_gfx_last_error(nat):
    lib = nat.lib
    rc = lib.gfx_align(None, 0, None, 0, None, 1, 0.0, 0.0, 1.0, None, None, None, 0, None)
    assert rc != 0 and b"positive" in lib.gfx_last_error()
    rc = lib.gfx_align(None, 0, None, 0, None, 1, 0.0, 1.0, -1.0, None, None, None, 0, None)
    assert rc != 0 and b"positive" in lib.gfx_last_error()
    rc = lib.gfx_align(None, 0, None, 0, None, 1, float("nan"), 1.0, 1.0, None, None, None, 0, None)
    assert rc != 0 and b"finite" in lib.gfx_last_error()
    rc = lib.gfx_align(None, 0, None, 0, None, -1, 0.0, 1.0, 1.0, None, None, None, 0, None)
    assert rc != 0 and b"bad sizes" in lib.gfx_last_error()
    rc = lib.gfx_align(None, 0, None, 0, None, 3, 0.0, 1.0, 1.0, None, None, None, 0, None)
    assert rc != 0 and b"null pointer" in lib.gfx_last_error()
    # nothing to do is not an error
    assert lib.gfx_align(None, 0, None, 0, None, 0, 0.0, 1.0, 1.0, None, None, None, 0, None) == 0
    small = lib.gfx_align_workspace_bytes(10, 0)
    assert lib.gfx_align_workspace_bytes(10, 4096) >= small + 10 * 4096 * 16
    assert lib.gfx_align_workspace_bytes(10, 100000) == lib.gfx_align_workspace_bytes(10, 4096)
    assert "align" in nat.STAGES


def _call(**kw):
    from ginfinity_b200.align import align_pairs
    args = dict(queries=np.zeros((10, 128), np.float16), targets=np.zeros((20, 128), np.float16),
                pairs=np.array([[0, 10, 0, 20]]), offset=0.5, gap_open=1.0, gap_extend=0.5)
    args.update(kw)
    return align_pairs(args.pop("queries"), args.pop("targets"), args.pop("pairs"), **args)


@pytest.mark.parametrize("kw, message", [
    (dict(queries=np.zeros((10, 64), np.float16)), r"\[rows, 128\]"),
    (dict(targets=np.zeros((20, 128), np.float32)), "float32"),
    (dict(queries=np.zeros((10, 128), np.float64)), "float16"),
    (dict(pairs=np.array([[0, 10, 0]])), r"\[P, 4\]"),
    (dict(pairs=np.array([[0.0, 10, 0, 20]])), "integer"),
    (dict(pairs=np.array([[0, 11, 0, 20]])), "outside the table"),
    (dict(pairs=np.array([[-1, 1, 0, 20]])), "outside the table"),
    (dict(pairs=np.array([[0, 10, 5, 16]])), "outside the table"),
    (dict(pairs=np.array([[0, 10, 0, -1]])), "length"),
    (dict(queries=np.zeros((5000, 128), np.float16), pairs=np.array([[0, 4097, 0, 20]])), "length"),
    (dict(gap_open=0.0), "positive"),
    (dict(gap_extend=-0.5), "positive"),
    (dict(offset=math.inf), "finite"),
    (dict(gap_open=1e39), "finite"),
    (dict(offset="0.5"), "real number"),
])
def test_align_pairs_validates_before_device_work(nat, kw, message):
    with pytest.raises((ValueError, TypeError), match=message):
        _call(**kw)


def test_align_pairs_refuses_non_finite_embeddings(nat):
    q = np.zeros((10, 128), np.float16)
    q[3, 7] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        _call(queries=q)
    t = np.zeros((20, 128), np.float16)
    t[0, 0] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        _call(targets=t)


def test_parameters_are_required_keywords(nat):
    from ginfinity_b200.align import align_pairs
    with pytest.raises(TypeError):
        align_pairs(np.zeros((1, 128), np.float16), np.zeros((1, 128), np.float16),
                    np.zeros((0, 4), np.int64))
    with pytest.raises(TypeError):
        align_pairs(np.zeros((1, 128), np.float16), np.zeros((1, 128), np.float16),
                    np.zeros((0, 4), np.int64), 0.5, 1.0, 0.5)
    import ginfinity_b200 as g
    assert g.align_pairs is align_pairs
