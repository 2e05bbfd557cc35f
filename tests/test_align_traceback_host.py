"""Alignment traceback (align_paths / gfx_align_trace) without a GPU: the
oracle's path against brute force and the hand-built ties, argument errors of
the C ABI, the Python layer's validation and the CIGAR formatting."""
import math
import shutil

import numpy as np
import pytest

from align_path_oracle import OP_D, OP_I, OP_M, align_fp32_path, dp_codes, path_score
from oracle.align_oracle import _dp, align_fp32
from test_align_host import brute_force, dyadic


def check_path(ops, qb, qe, tb, te):
    """A valid path: starts and ends with M and consumes exactly the region."""
    ops = np.asarray(ops)
    assert ops[0] == OP_M and ops[-1] == OP_M
    assert (ops == OP_M).sum() + (ops == OP_I).sum() == qe - qb
    assert (ops == OP_M).sum() + (ops == OP_D).sum() == te - tb
    assert set(np.unique(ops).tolist()) <= {OP_M, OP_I, OP_D}


@pytest.mark.parametrize("seed", range(40))
def test_oracle_path_matches_brute_force_on_small_dyadic_inputs(seed):
    rng = np.random.default_rng(seed)
    n, m = rng.integers(1, 5, size=2)
    S = dyadic(rng, (n, m))
    th, go, ge = 0.25 * rng.integers(0, 3), 0.25 * rng.integers(1, 5), 0.25 * rng.integers(1, 3)
    res, ops = align_fp32_path(S, th, go, ge)
    assert res == align_fp32(S, th, go, ge)
    score, qb, qe, tb, te = res
    if score == 0:
        assert len(ops) == 0
        return
    check_path(ops, qb, qe, tb, te)
    assert path_score(S.astype(np.float64), ops, (qb, tb), th, go, ge) == brute_force(S.astype(np.float64), th, go, ge)
    f32 = path_score(S, ops, (qb, tb), th, go, ge)
    assert f32.dtype == np.float32 and f32.tobytes() == np.float32(score).tobytes()


def test_code_recording_dp_is_the_score_oracle_dp():
    rng = np.random.default_rng(3)
    for dt in (np.float32, np.float64):
        for _ in range(20):
            n, m = rng.integers(1, 30, size=2)
            S = rng.standard_normal((n, m)).astype(dt)
            H, sH, _ = dp_codes(S, 0.3, 1.1, 0.35)
            H0, sH0 = _dp(S, 0.3, 1.1, 0.35)
            assert H.tobytes() == H0.tobytes() and (sH == sH0).all()


def test_paths_on_rounding_parameters_rescore_bit_for_bit():
    rng = np.random.default_rng(7)
    for _ in range(30):
        n, m = rng.integers(5, 40, size=2)
        S = rng.standard_normal((n, m)).astype(np.float32)
        res, ops = align_fp32_path(S, 0.3, 1.1, 0.35)
        if res[0] == 0:
            continue
        check_path(ops, *res[1:])
        assert path_score(S, ops, (res[1], res[3]), 0.3, 1.1, 0.35).tobytes() == np.float32(res[0]).tobytes()


def test_diagonal_wins_over_equal_gaps():
    S = np.array([[2.0, 1.0], [1.0, -1.0]], np.float32)
    res, ops = align_fp32_path(S, 0.0, 1.0, 1.0)
    assert res == (2.0, 0, 1, 0, 1) and ops.tolist() == [OP_M]
    # on a path: H(1,1) = 1.5 - 1 = 0.5 from the diagonal, and E(1,1) = H(1,0) - 0.5 and
    # F(1,1) = H(0,1) - 0.5 are 0.5 too; the diagonal wins, so the path is three M steps
    S = np.array([[1.5, -1.5, 2.0], [-1.5, -1.0, -2.0], [0.5, -1.0, 2.0]], np.float32)
    H, _, codes = dp_codes(S, 0.0, 0.5, 0.5)
    assert H[2, 2] == H[2, 1] - 0.5 == H[1, 2] - 0.5 == 0.5 and codes[1, 1] & 3 == 1
    res, ops = align_fp32_path(S, 0.0, 0.5, 0.5)
    assert res == (2.5, 0, 3, 0, 3) and ops.tolist() == [OP_M, OP_M, OP_M]


def test_e_wins_over_equal_f_and_diagonal_start_rule():
    # the cells of test_align_host's matrix, extended by a column that makes (1,2) the end:
    # H(1,1) = 0.5 from the diagonal (a new start, since H(0,0) = 0)
    S = np.array([[0.0, 2.0, 0.0], [2.0, 0.5, 9.0]], np.float32)
    res, ops = align_fp32_path(S, 0.0, 1.5, 1.0)
    # (1,2): diagonal from H(0,1) = 2 gives 11; E from H(1,1) = 0.5 gives -1
    assert res == (11.0, 0, 2, 1, 3) and ops.tolist() == [OP_M, OP_M]
    # without the diagonal at (1,1), E and F tie there at 0.5; E (the left one) wins, and the
    # alignment ending at (1,1) is "M at (1,0), then a D step"
    S = np.array([[0.0, 2.0, 0.0], [2.0, -8.0, 0.0]], np.float32)
    H, sH, codes = dp_codes(S, 0.0, 1.5, 1.0)
    assert H[2, 2] == 0.5 and sH[2, 2] == (1 << 16) | 0
    assert codes[1, 1] & 3 == 2                       # H(1,1) from E
    # the start rule: a diagonal step from H = 0 starts the alignment at that cell
    S = np.array([[-5.0, -5.0], [-5.0, 3.0]], np.float32)
    res, ops = align_fp32_path(S, 0.0, 1.0, 1.0)
    assert res == (3.0, 1, 2, 1, 2) and ops.tolist() == [OP_M]


def test_opening_wins_over_extending():
    # the row of test_align_host: at (0,2) opening from H(0,1) and extending E(0,1) tie at 1
    S = np.array([[3.0, 2.0, -9.0, 9.0]], np.float32)
    codes = dp_codes(S, 0.0, 1.0, 1.0)[2]
    assert codes[0, 2] & 4                            # E(0,2) opened
    # the same row above a cell that ends the alignment at (1,3) through H(0,2) = E(0,2): the
    # gap is taken as opened at (0,1), so the path is M (0,1), D (0,2), M (1,3), not from (0,0)
    S = np.array([[3.0, 2.0, -9.0, -9.0], [-9.0, -9.0, -9.0, 9.0]], np.float32)
    res, ops = align_fp32_path(S, 0.0, 1.0, 1.0)
    assert res == (10.0, 0, 2, 1, 4) and ops.tolist() == [OP_M, OP_D, OP_M]
    # rows instead of columns: an I step, F opened
    res, ops = align_fp32_path(S.T.copy(), 0.0, 1.0, 1.0)
    assert res == (10.0, 1, 4, 0, 2) and ops.tolist() == [OP_M, OP_I, OP_M]
    # a longer gap: open then extend, both kinds in one path
    S = np.array([[5, -9, -9, -9, -9], [-9, -9, -9, -9, 9], [-9, -9, -9, -9, -9], [-9, -9, -9, -9, 9]],
                 np.float32)
    res, ops = align_fp32_path(S, 0.0, 1.0, 0.5)
    check_path(ops, *res[1:])
    assert path_score(S, ops, (res[1], res[3]), 0.0, 1.0, 0.5).tobytes() == np.float32(res[0]).tobytes()


def test_path_score_charges_opening_after_the_other_gap_kind():
    S = np.zeros((3, 3), np.float32)
    S[0, 0] = S[2, 2] = 8.0
    v = path_score(S, [OP_M, OP_D, OP_I, OP_M], (0, 0), 0.0, 1.0, 0.25)
    assert v == np.float32(8 - 1 - 1 + 8)
    S = np.zeros((2, 4), np.float32)
    S[0, 0] = S[1, 3] = 8.0
    v = path_score(S, [OP_M, OP_D, OP_D, OP_M], (0, 0), 0.0, 1.0, 0.25)
    assert v == np.float32(8 - 1 - 0.25 + 8)


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


def test_gfx_align_trace_argument_errors_surface_through_gfx_last_error(nat):
    lib = nat.lib

    def call(num_pairs, offset, go, ge, ops=None, offs=None, lens=None, ws=None, ws_bytes=0, pairs=None,
             score=None, coords=None):
        return lib.gfx_align_trace(None, 0, None, 0, pairs, num_pairs, offset, go, ge, score, coords, ops,
                                   offs, lens, ws, ws_bytes, None)

    assert call(1, 0.0, 0.0, 1.0) != 0 and b"positive" in lib.gfx_last_error()
    assert call(1, 0.0, 1.0, -1.0) != 0 and b"positive" in lib.gfx_last_error()
    assert call(1, float("nan"), 1.0, 1.0) != 0 and b"finite" in lib.gfx_last_error()
    assert call(-1, 0.0, 1.0, 1.0) != 0 and b"bad sizes" in lib.gfx_last_error()
    assert call(3, 0.0, 1.0, 1.0) != 0 and b"null pointer" in lib.gfx_last_error()
    assert lib.gfx_last_error().startswith(b"gfx_align_trace:")
    # the order of gfx_align: sizes, then parameters
    assert call(-1, float("nan"), 0.0, 1.0) != 0 and b"bad sizes" in lib.gfx_last_error()
    # every pointer of gfx_align given, the trace outputs missing (addresses only, never read)
    fake = 1 << 20
    kw = dict(pairs=fake, score=fake, coords=fake, ws=fake, ws_bytes=1 << 40)
    for missing in ("ops", "offs", "lens"):
        given = {k: fake for k in ("ops", "offs", "lens") if k != missing}
        assert call(3, 0.0, 1.0, 1.0, **given, **kw) != 0 and b"null pointer" in lib.gfx_last_error()
    # a workspace below the fixed part is refused before any device work
    small = lib.gfx_align_trace_workspace_bytes(3, 0)
    kw["ws_bytes"] = small - 1
    assert call(3, 0.0, 1.0, 1.0, ops=fake, offs=fake, lens=fake, **kw) != 0
    assert b"workspace too small" in lib.gfx_last_error()
    # nothing to do is not an error
    assert call(0, 0.0, 1.0, 1.0) == 0


def test_gfx_align_trace_workspace_bytes(nat):
    f = nat.lib.gfx_align_trace_workspace_bytes
    assert f(10, 0) < f(11, 0) and f(10, 0) < f(10, 1) and f(10, 1) < f(10, 1 << 20)
    assert f(-5, -5) == f(0, 0) and f(10, -1) == f(10, 0)
    # hand-computed batches: (q_len, t_len) -> q_len * ceil(t_len / 32) * 16 bytes of codes
    for batch, codes in (([(1, 1)], 16), ([(100, 32), (100, 33)], 100 * 16 + 100 * 32),
                         ([(4096, 4096)], 8 << 20), ([(0, 50), (7, 0), (3, 65)], 3 * 3 * 16)):
        got = sum(q * ((t + 31) // 32) * 16 for q, t in batch)
        assert got == codes
        assert f(len(batch), codes) - f(len(batch), 0) == codes
    # the fixed part covers the score pass's workspace for any target length
    assert f(10, 0) >= nat.lib.gfx_align_workspace_bytes(10, 4096)
    assert f(1000, 0) >= nat.lib.gfx_align_workspace_bytes(1000, 4096) + 1000 * 8


def _paths(**kw):
    from ginfinity_b200.align import align_paths
    args = dict(queries=np.zeros((10, 128), np.float16), targets=np.zeros((20, 128), np.float16),
                pairs=np.array([[0, 10, 0, 20]]), offset=0.5, gap_open=1.0, gap_extend=0.5)
    args.update(kw)
    return align_paths(args.pop("queries"), args.pop("targets"), args.pop("pairs"), **args)


def _pairs_call(**kw):
    from ginfinity_b200.align import align_pairs
    args = dict(queries=np.zeros((10, 128), np.float16), targets=np.zeros((20, 128), np.float16),
                pairs=np.array([[0, 10, 0, 20]]), offset=0.5, gap_open=1.0, gap_extend=0.5)
    args.update(kw)
    return align_pairs(args.pop("queries"), args.pop("targets"), args.pop("pairs"), **args)


def _nonfinite():
    q = np.zeros((10, 128), np.float16)
    q[3, 7] = np.inf
    return q


@pytest.mark.parametrize("kw", [
    dict(queries=np.zeros((10, 64), np.float16)),
    dict(targets=np.zeros((20, 128), np.float32)),
    dict(queries=np.zeros((10, 128), np.float64)),
    dict(pairs=np.array([[0, 10, 0]])),
    dict(pairs=np.array([[0.0, 10, 0, 20]])),
    dict(pairs=np.array([[0, 11, 0, 20]])),
    dict(pairs=np.array([[-1, 1, 0, 20]])),
    dict(pairs=np.array([[0, 10, 5, 16]])),
    dict(pairs=np.array([[0, 10, 0, -1]])),
    dict(queries=np.zeros((5000, 128), np.float16), pairs=np.array([[0, 4097, 0, 20]])),
    dict(gap_open=0.0),
    dict(gap_extend=-0.5),
    dict(offset=math.inf),
    dict(gap_open=1e39),
    dict(offset="0.5"),
    dict(queries=_nonfinite()),
    dict(device="cpu"),
])
def test_align_paths_validates_like_align_pairs(nat, kw):
    with pytest.raises((ValueError, TypeError)) as want:
        _pairs_call(**kw)
    with pytest.raises(want.type) as got:
        _paths(**kw)
    assert str(got.value) == str(want.value)


def test_align_paths_parameters_are_required_keywords(nat):
    from ginfinity_b200.align import align_paths
    z = np.zeros((1, 128), np.float16)
    with pytest.raises(TypeError):
        align_paths(z, z, np.zeros((0, 4), np.int64))
    with pytest.raises(TypeError):
        align_paths(z, z, np.zeros((0, 4), np.int64), 0.5, 1.0, 0.5)
    import ginfinity_b200 as g
    assert g.align_paths is align_paths
    assert g.AlignmentPaths.__name__ == "AlignmentPaths"
    with pytest.raises(ValueError, match="float32"):
        align_paths(z.astype(np.float32), z, np.zeros((0, 4), np.int64), offset=0.5, gap_open=1.0,
                    gap_extend=0.5)


def test_cigars_of_hand_built_paths(nat):
    torch = pytest.importorskip("torch")
    from ginfinity_b200.align import AlignmentPaths
    M, I, D = OP_M, OP_I, OP_D
    paths = [[M] * 12 + [I] * 2 + [M] * 30 + [D] + [M] * 5, [], [M], [M, D, I, M], [M, I, M, I, M]]
    ops = np.concatenate([np.array(p, np.uint8) for p in paths] + [np.zeros(0, np.uint8)])
    lens = np.array([len(p) for p in paths], np.int32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
    # slots with spare room after each path, as align_paths leaves them
    spaced = np.zeros(len(ops) + 3 * len(paths), np.uint8)
    offs2 = offs + 3 * np.arange(len(paths))
    for p, (o, n) in enumerate(zip(offs, lens)):
        spaced[offs2[p]:offs2[p] + n] = ops[o:o + n]
        spaced[offs2[p] + n:offs2[p] + n + 3] = 7
    want = ["12M2I30M1D5M", "", "1M", "1M1D1I1M", "1M1I1M1I1M"]
    for o, data in ((offs, ops), (offs2, spaced)):
        paths_obj = AlignmentPaths(torch.from_numpy(data), torch.from_numpy(o), torch.from_numpy(lens))
        assert paths_obj.cigars() == want
    empty = AlignmentPaths(torch.zeros(0, dtype=torch.uint8), torch.zeros(0, dtype=torch.int64),
                           torch.zeros(0, dtype=torch.int32))
    assert empty.cigars() == []
