"""CPU checks of the float32 search: the fp32-row oracle against float64,
the planted constructions of tests/test_gpu_search_f32.py, the workspace
layout of gfx_topk_f32 and its argument errors, and (where cuobjdump is
installed) the instructions of the split-fp16 scan."""
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from f32_oracle import (exact_scores_f32, fma32, fp16_collisions, near_tie_rows, topk_exact_f32,
                        unit_rows32)
from oracle import gine_oracle as O

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "ginfinity_b200" / "libgfx.so"


def test_fma32_is_correctly_rounded():
    """Against exact rational arithmetic on values where double rounding of the
    plain float64 sum would be wrong."""
    from fractions import Fraction
    rng = np.random.default_rng(0)
    a = rng.normal(size=4000).astype(np.float32)
    b = (rng.normal(size=4000) * 2.0 ** rng.integers(-40, 0, 4000)).astype(np.float32)
    acc = rng.normal(size=4000).astype(np.float32)
    # ties of the float64 sum: a*b = 2^-24 (1 + 2^-36), half an fp32 ulp of 1 plus a term
    # below float64's resolution, so 1 + a*b rounds to the fp32 midpoint 1 + 2^-24 in float64
    sign = np.where(np.arange(8) < 4, 1.0, -1.0).astype(np.float32)
    acc[:8] = sign
    a[:8] = sign * np.float32(2.0 ** -24 * (1 + 2.0 ** -12))
    b[:8] = np.float32(1 - 2.0 ** -12 + 2.0 ** -24)
    f64_sum = acc[:8].astype(np.float64) + a[:8].astype(np.float64) * b[:8]
    assert np.all(f64_sum == sign.astype(np.float64) * (1 + 2.0 ** -24))
    got = fma32(a, b, acc)
    assert np.all(got[:8] == sign * np.float32(1 + 2.0 ** -23))
    for i in range(len(a)):
        exact = Fraction(float(acc[i])) + Fraction(float(a[i])) * Fraction(float(b[i]))
        lo = np.float32(float(exact))
        cands = [lo, np.nextafter(lo, np.float32(np.inf)), np.nextafter(lo, np.float32(-np.inf))]
        best = min(cands, key=lambda c: (abs(Fraction(float(c)) - exact),
                                         int(np.float32(c).view(np.uint32)) & 1))
        assert got[i] == best, i


def test_f32_oracle_equals_the_fp16_oracle_on_fp16_values():
    """On rows and queries that fp16 represents exactly the two oracles agree."""
    rng = np.random.default_rng(1)
    q = unit_rows32(rng, 6).astype(np.float16)
    x = unit_rows32(rng, 50).astype(np.float16)
    for metric in ("cosine", "l2"):
        np.testing.assert_array_equal(exact_scores_f32(q.astype(np.float32), x.astype(np.float32), metric),
                                      O.exact_scores_fp32(q, x, metric))


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_f32_oracle_agrees_with_float64_where_gaps_are_resolvable(metric):
    rng = np.random.default_rng(2)
    q, x, k = unit_rows32(rng, 40), unit_rows32(rng, 3000), 10
    got_s, got_i = topk_exact_f32(q, x, k, metric)
    if metric == "cosine":
        f64 = q.astype(np.float64) @ x.astype(np.float64).T
    else:
        f64 = -((q.astype(np.float64)[:, None] - x.astype(np.float64)[None]) ** 2).sum(-1)
    order = np.argsort(-f64, axis=1, kind="stable")[:, :k + 1]
    want = np.take_along_axis(f64, order, 1)
    np.testing.assert_allclose(got_s, want[:, :k], rtol=0, atol=2e-6)
    clear = np.all(want[:, :-1] - want[:, 1:] > 1e-5, axis=1)
    assert clear.mean() > 0.9
    np.testing.assert_array_equal(got_i[clear], order[clear, :k])


@pytest.mark.parametrize("metric", ["cosine", "l2"])
def test_fp16_collisions_collide_in_fp16_and_are_strict_in_fp32(metric):
    rng = np.random.default_rng(3)
    base = unit_rows32(rng, 1)[0].astype(np.float16).astype(np.float32)
    rows = fp16_collisions(rng, base, 30)
    assert len(np.unique(rows, axis=0)) == 30                          # distinct in fp32
    assert len(np.unique(rows.astype(np.float16), axis=0)) == 1        # one row in fp16
    s = exact_scores_f32(base[None], rows, metric)[0]
    assert len(np.unique(s)) == 30                                     # a strict fp32 order ...
    order = np.argsort(-s.astype(np.float64), kind="stable")
    assert not np.array_equal(order, np.arange(30))                    # ... that is not index order
    s16 = O.exact_scores_fp32(base[None].astype(np.float16), rows.astype(np.float16), metric)[0]
    assert len(np.unique(s16)) == 1                                    # fp16: all tie


def test_near_tie_rows_are_below_the_split_margin():
    """The rows of the near-tie GPU case differ in score by far less than the
    split scan's margin (2^-13 |q| N_max), yet their fp32 scores are distinct."""
    rng = np.random.default_rng(4)
    q = unit_rows32(rng, 1)[0]
    rows = near_tie_rows(rng, q, 40)
    s = exact_scores_f32(q[None], rows, "cosine")[0].astype(np.float64)
    assert s.max() - s.min() < 2.0 ** -13 / 4
    assert len(np.unique(s)) > 25


# ---------------- the C ABI without a GPU ---------------------------------------------------


@pytest.fixture(scope="module")
def nat():
    try:
        from ginfinity_b200 import _native
    except ImportError:
        pytest.skip("libgfx.so is not built")
    return _native


def f32_plan_bytes(Q, D, k):
    """gfx_topk_f32's workspace: gfx_topk's regions laid out for 128-query tiles,
    then the [Q, 256] fp16 image of the queries."""
    up = lambda v: -(-v // 256) * 256  # noqa: E731
    tiles_q, tiles_db = -(-Q // 128), -(-D // 128)
    segs = -(-8 * 148 // tiles_q) if tiles_q < 8 * 148 else 1
    segs = min(segs, max(tiles_db // 16, 1))
    per_seg = -(-tiles_db // segs) if tiles_db else 1
    segs = -(-tiles_db // per_seg) if tiles_db else 1
    kc = min((k + 7) & ~3, 28)
    cand = segs * tiles_q * 128 * kc
    need = 256 + up(4 * Q) + 2 * up(4 * cand) + up(4 * tiles_db * 128)
    if tiles_db >= 8 * 128:
        need += 2 * up(4 * tiles_q * 128 * kc)
    return need + up(Q * 512)


@pytest.mark.parametrize("Q,D,k", [(1, 40_000, 1), (300, 20_000, 24), (2048, 1_000_000, 10),
                                   (100_000, 1_000_000, 10), (5, 0, 3)])
def test_f32_workspace_holds_every_region(nat, Q, D, k):
    assert nat.lib.gfx_topk_f32_workspace_bytes(Q, D, k) == f32_plan_bytes(Q, D, k)
    assert nat.lib.gfx_topk_f32_workspace_bytes(0, D, k) == 256


def test_f32_argument_errors(nat):
    lib = nat.lib
    cases = [
        (lambda: lib.gfx_topk_f32(None, 1, None, None, 1, 64, 3, 0, 0, None, None, None, 0, None), b"dim = 128"),
        (lambda: lib.gfx_topk_f32(None, 1, None, None, 1, 128, 25, 0, 0, None, None, None, 0, None), b"k must be"),
        (lambda: lib.gfx_topk_f32(None, 1, None, None, 1, 128, 3, 2, 0, None, None, None, 0, None), b"metric"),
        (lambda: lib.gfx_topk_f32(None, -1, None, None, 1, 128, 3, 0, 0, None, None, None, 0, None), b"bad sizes"),
        (lambda: lib.gfx_topk_f32(None, 1, None, None, 1, 128, 3, 0, 0, None, None, None, 0, None), b"null pointer"),
        (lambda: lib.gfx_topk_f32(8, 1, 16, 32, 1, 128, 3, 0, 0, 64, 64, None, 0, None), b"16-byte aligned"),
        (lambda: lib.gfx_topk_f32(16, 1, 16, 32, 1, 128, 3, 0, 0, 64, 64, None, 0, None), b"workspace too small"),
        (lambda: lib.gfx_topk_f32_prepare(None, -1, None, None), b"bad sizes"),
        (lambda: lib.gfx_topk_f32_prepare(None, 4, None, None), b"null pointer"),
        (lambda: lib.gfx_topk_f32_prepare(16, 4, 8, None), b"16-byte aligned"),
    ]
    for call, message in cases:
        rc = call()
        assert rc != 0 and message in lib.gfx_last_error(), message
    assert lib.gfx_topk_f32(None, 0, None, None, 0, 128, 3, 0, 0, None, None, None, 0, None) == 0
    assert lib.gfx_topk_f32_prepare(None, 0, None, None) == 0


def _kernel_sass(sass, needle):
    parts = sass.split("Function : ")
    body = [p for p in parts if needle in p.split("\n", 1)[0]]
    assert body, needle
    return body[0]


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump is not installed here")
def test_split_scan_issues_24_mmas_per_tile_from_uniform_registers(nat):
    """Three kind::f16 MMAs (hi.hi, hi.lo, lo.hi) per 16-wide K step, 8 K steps per
    128-row database tile; the elected-lane issuers keep their operands in
    uniform registers (no ELECT / R2UR.BROADCAST loop around each MMA)."""
    sass = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True).stdout
    for metric in (0, 1):
        scan = _kernel_sass(sass, f"split_search_kernelILi{metric}E")
        assert len(re.findall(r"\bUTCHMMA\b", scan)) == 24
        assert scan.count("R2UR.BROADCAST") <= 2 * scan.count("UTMALDG")
        assert "HMMA." not in scan.replace("UTCHMMA", "")
