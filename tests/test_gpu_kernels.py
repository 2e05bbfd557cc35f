"""GPU parity tests, kernel by kernel, through the C ABI (ctypes -> libgfx.so).

Oracle: oracle/gine_oracle.py (NumPy restatement of the reference, pinned to
the reference's own outputs by tests/test_oracle_golden.py).
Bars: integer/index work bit-exact; fp32 path |err| <= 2e-5 on O(10) values;
fp16-storage path compared with the oracle run with the same fp16 storage
points (tolerances written at each assert).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import gine_oracle as O  # noqa: E402
from helpers import random_records  # noqa: E402


@pytest.fixture(scope="module")
def nat():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ginfinity_b200 import _native
    return _native


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _up(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def device_csr(nat, dev, edge_index, edge_types, n, base=0):
    e = edge_index.shape[1]
    ei, et = _up(edge_index, dev), _up(edge_types, dev)
    row_ptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
    col_src = torch.empty(max(e, 1), dtype=torch.int32, device=dev)
    col_type = torch.empty(max(e, 1), dtype=torch.uint8, device=dev)
    need = nat.lib.gfx_csr_workspace_bytes(n, e)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    nat.check(nat.lib.gfx_csr_build(
        ei[0].data_ptr() if e else None, ei[1].data_ptr() if e else None,
        et.data_ptr() if e else None, n, e, base, row_ptr.data_ptr(),
        col_src.data_ptr(), col_type.data_ptr(), ws.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    return row_ptr, col_src[:e], col_type[:e]


# ---------------------------------------------------------------- K0: CSR
@pytest.mark.parametrize("seed,count", [(1, 1), (2, 40), (3, 600)])
def test_csr_matches_stable_argsort(nat, dev, seed, count):
    import ginfinity_b200 as g
    shard = g.GraphBuilder().build_shard(random_records(seed, count))
    rp, cs, ct = device_csr(nat, dev, shard.edge_index, shard.edge_types,
                            shard.node_count)
    erp, ecs, ect = O.csr_by_destination(shard.edge_index, shard.edge_types,
                                         shard.node_count)
    assert np.array_equal(rp.cpu().numpy(), erp)          # bit-exact
    assert np.array_equal(cs.cpu().numpy(), ecs)
    assert np.array_equal(ct.cpu().numpy(), ect)
    # run-to-run determinism (the scatter pass uses atomics internally)
    rp2, cs2, ct2 = device_csr(nat, dev, shard.edge_index, shard.edge_types,
                               shard.node_count)
    assert torch.equal(cs, cs2) and torch.equal(ct, ct2) and torch.equal(rp, rp2)


def test_csr_arbitrary_graph_duplicates_self_loops_hubs(nat, dev):
    """Shards may hold any valid edge list: duplicates, self loops, isolated
    nodes and hub nodes far above the small-row threshold."""
    rng = np.random.default_rng(5)
    n, e = 5000, 60000
    src = rng.integers(0, n, e).astype(np.int32)
    dst = rng.integers(0, n, e).astype(np.int32)
    dst[:9000] = 17                      # hub: 9000 in-edges
    dst[9000:9100] = 4999
    src[100:200] = dst[100:200]          # self loops
    src[300:400], dst[300:400] = src[200:300], dst[200:300]   # duplicates
    dst[dst == 123] = 124                # isolated node
    typ = rng.integers(0, 10, e).astype(np.uint8)
    ei = np.stack([src, dst])
    rp, cs, ct = device_csr(nat, dev, ei, typ, n)
    erp, ecs, ect = O.csr_by_destination(ei, typ, n)
    assert np.array_equal(rp.cpu().numpy(), erp)
    assert np.array_equal(cs.cpu().numpy(), ecs)
    assert np.array_equal(ct.cpu().numpy(), ect)


def test_csr_rebases_a_shard_slice(nat, dev):
    import ginfinity_b200 as g
    shard = g.GraphBuilder().build_shard(random_records(9, 30))
    a, b = 7, 19
    n0, n1 = int(shard.node_ptr[a]), int(shard.node_ptr[b])
    e0, e1 = int(shard.edge_ptr[a]), int(shard.edge_ptr[b])
    rp, cs, ct = device_csr(nat, dev, shard.edge_index[:, e0:e1],
                            shard.edge_types[e0:e1], n1 - n0, base=n0)
    sub = shard.slice(a, b)              # host rebasing (reference semantics)
    erp, ecs, ect = O.csr_by_destination(sub.edge_index, sub.edge_types,
                                         sub.node_count)
    assert np.array_equal(rp.cpu().numpy(), erp)
    assert np.array_equal(cs.cpu().numpy(), ecs)
    assert np.array_equal(ct.cpu().numpy(), ect)


def test_csr_empty_edges(nat, dev):
    rp, cs, ct = device_csr(nat, dev, np.zeros((2, 0), np.int32),
                            np.zeros(0, np.uint8), 3)
    assert rp.cpu().tolist() == [0, 0, 0, 0]


# ------------------------------------------------------------ K4: packing
def device_pack(nat, dev, node_ptr, edge_ptr, max_nodes, max_edges):
    B = node_ptr.shape[0] - 1
    nptr, eptr = _up(node_ptr, dev), _up(edge_ptr, dev)
    nxt = torch.empty(B, dtype=torch.int64, device=dev)
    bounds = torch.empty(B + 1, dtype=torch.int64, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    nat.check(nat.lib.gfx_pack_microbatches(
        nptr.data_ptr(), eptr.data_ptr(), B, max_nodes, max_edges,
        nxt.data_ptr(), bounds.data_ptr(), count.data_ptr(), _stream()))
    torch.cuda.synchronize()
    return bounds[:int(count.item())].cpu().numpy()


@pytest.mark.parametrize("limits", [(60_000, 300_000), (700, 3000), (1000, 4600),
                                    (100_000, 2000), (450, 100_000)])
def test_pack_matches_reference_greedy(nat, dev, limits):
    import ginfinity_b200 as g
    shard = g.GraphBuilder().build_shard(random_records(11, 300))
    lengths = np.diff(shard.node_ptr).tolist()
    ecounts = np.diff(shard.edge_ptr).tolist()
    if max(lengths) > limits[0] or max(ecounts) > limits[1]:
        pytest.skip("limits below the largest graph are rejected on the host")
    want = O.pack_microbatches(lengths, ecounts, *limits)
    got = device_pack(nat, dev, shard.node_ptr, shard.edge_ptr, *limits)
    assert np.array_equal(got, want)


def test_pack_golden_boundaries_from_the_reference(nat, dev, golden_meta, golden_shard):
    for case in golden_meta["packing"]:
        if isinstance(case["bounds"], dict):
            continue
        got = device_pack(nat, dev, golden_shard.node_ptr, golden_shard.edge_ptr,
                          case["max_batch_nodes"], case["max_batch_edges"])
        assert got.tolist() == case["bounds"]


# ------------------------------------------------------------- core rows
def test_core_row_map(nat, dev):
    rng = np.random.default_rng(3)
    roles = (rng.random(10_007) < 0.3).astype(np.uint8)
    r = _up(roles, dev)
    out = torch.empty(roles.shape[0], dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    need = nat.lib.gfx_core_rows_workspace_bytes(roles.shape[0])
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    nat.check(nat.lib.gfx_core_rows(r.data_ptr(), roles.shape[0], out.data_ptr(),
                                    cnt.data_ptr(), ws.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    want = np.where(roles == 0, np.cumsum(roles == 0) - 1, -1)
    assert np.array_equal(out.cpu().numpy(), want)
    assert int(cnt.item()) == int((roles == 0).sum())


# ----------------------------------------------------- float stages
@pytest.fixture(scope="module")
def problem(nat, dev, synthetic_state):
    import ginfinity_b200 as g
    from ginfinity_b200.weights import fold
    shard = g.GraphBuilder().build_shard(random_records(21, 25))   # ~5k nodes
    fw = O.fold_state(synthetic_state)
    handle = nat.model_create(fold(synthetic_state))
    rp, cs, ct = device_csr(nat, dev, shard.edge_index, shard.edge_types,
                            shard.node_count)
    erp, ecs, ect = O.csr_by_destination(shard.edge_index, shard.edge_types,
                                         shard.node_count)
    y32, keep32 = O.forward_folded(fw, shard.node_features, erp, ecs, ect,
                                   return_intermediates=True)
    y16, keep16 = O.forward_folded(fw, shard.node_features, erp, ecs, ect,
                                   half_storage=True, return_intermediates=True)
    # the fused layer kernels' arithmetic: fp16 sum chain, fp16 self term, fp16 residual add
    y16s, keep16s = O.forward_folded(fw, shard.node_features, erp, ecs, ect, half_storage=True,
                                     half_sums=True, return_intermediates=True)
    yield dict(shard=shard, fw=fw, handle=handle, csr=(rp, cs, ct),
               y32=y32, keep32=keep32, y16=y16, keep16=keep16, y16s=y16s, keep16s=keep16s)
    nat.model_destroy(handle)


def _buf(n, code, dev):
    return torch.empty((n, 128), dtype=torch.float16 if code == 0 else torch.float32,
                       device=dev)


def test_input_linear(nat, dev, problem):
    x = _up(problem["shard"].node_features, dev)
    n = x.shape[0]
    for code, key, tol in ((1, "keep32", 2e-6), (0, "keep16", 0.0)):
        h = _buf(n, code, dev)
        nat.check(nat.lib.gfx_input_linear(problem["handle"], x.data_ptr(), n,
                                           h.data_ptr(), code, _stream()))
        torch.cuda.synchronize()
        want = problem[key]["h0"]
        got = h.float().cpu().numpy()
        if code == 0:   # fp16 storage: at most one fp16 ulp from a 7-term fp32 sum
            assert np.abs(got - want).max() <= 2 ** -10 * np.abs(want).max()
        else:
            assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("skip,count", [(1, 1), (1, 2), (2, 5), (3, 1001), (0, 1003), (5, 4096)])
def test_input_linear_unaligned_views_and_tails(nat, dev, problem, skip, count):
    """The vectorised kernel needs 16-byte aligned feature rows; a view that
    starts at an arbitrary node (what a chunk of a shard is) goes through the
    scalar lead-in, and sizes that are not a multiple of 4 through the tail."""
    x = _up(problem["shard"].node_features, dev)
    for code in (0, 1):
        full = _buf(x.shape[0], code, dev)
        nat.check(nat.lib.gfx_input_linear(problem["handle"], x.data_ptr(), x.shape[0],
                                           full.data_ptr(), code, _stream()))
        part = _buf(count, code, dev)
        nat.check(nat.lib.gfx_input_linear(problem["handle"], x[skip:].data_ptr(), count,
                                           part.data_ptr(), code, _stream()))
        torch.cuda.synchronize()
        assert torch.equal(part, full[skip:skip + count])


@pytest.mark.parametrize("code", [1, 0])
def test_aggregate_layer0(nat, dev, problem, code):
    """K1 against the oracle's z0 given the oracle's h0 as input."""
    keep = problem["keep32" if code == 1 else "keep16"]
    rp, cs, ct = problem["csr"]
    n = keep["h0"].shape[0]
    h = _up(keep["h0"], dev).to(torch.float32 if code == 1 else torch.float16)
    z = _buf(n, code, dev)
    nat.check(nat.lib.gfx_aggregate(problem["handle"], 0, h.data_ptr(), rp.data_ptr(),
                                    cs.data_ptr(), ct.data_ptr(), n, z.data_ptr(),
                                    code, _stream()))
    torch.cuda.synchronize()
    got, want = z.float().cpu().numpy(), keep["z0"]
    scale = np.abs(want).max()
    # fp32: same sums in the same order up to fma contraction; fp16: one
    # rounding of the stored result
    tol = 1e-6 * scale if code == 1 else 2 ** -10 * scale
    assert np.abs(got - want).max() <= tol
    # determinism
    z2 = _buf(n, code, dev)
    nat.check(nat.lib.gfx_aggregate(problem["handle"], 0, h.data_ptr(), rp.data_ptr(),
                                    cs.data_ptr(), ct.data_ptr(), n, z2.data_ptr(),
                                    code, _stream()))
    torch.cuda.synchronize()
    assert torch.equal(z, z2)


@pytest.mark.parametrize("n", [1, 3, 31, 33, 1000, 4099])
def test_aggregate_irregular_rows(nat, dev, problem, n):
    """K1 on rows the builder never produces: empty rows, rows longer than the
    quarter-warp kernel's straight-line window (5) and than its 8 fetched
    edges, self loops, duplicate edges, and node counts that leave quarters
    of the last warp without a node.  fp16 storage: bit-identical to the
    half-warp kernel's formula restated in NumPy (fp16 messages, fp32 sum in
    CSR order, one rounding of the result)."""
    rng = np.random.default_rng(100 + n)
    deg = rng.choice([0, 1, 2, 4, 5, 6, 8, 9, 17, 40], size=n,
                     p=[.1, .1, .1, .2, .2, .1, .05, .05, .05, .05])
    dst = np.repeat(np.arange(n), deg)
    src = rng.integers(0, n, size=dst.shape[0])
    src[::7] = dst[::7]                                  # self loops
    order = rng.permutation(dst.shape[0])                # unsorted input
    ei = np.stack([src[order], dst[order]]).astype(np.int32)
    et = rng.integers(0, 10, size=dst.shape[0]).astype(np.uint8)
    rp, cs, ct = device_csr(nat, dev, ei, et, n)
    erp, ecs, ect = O.csr_by_destination(ei, et, n)
    h = (rng.standard_normal((n, 128)) * 3).astype(np.float16)
    fw = problem["fw"]
    q = lambda a: a.astype(np.float16).astype(np.float32)   # noqa: E731
    hf = h.astype(np.float32)
    m = q(np.maximum(hf[ecs.astype(np.int64)] + q(fw["table"][1])[ect.astype(np.int64)], 0))
    agg = np.zeros_like(hf)
    np.add.at(agg, np.repeat(np.arange(n), np.diff(erp)), m)
    want = (np.float32(fw["eps1"][1]) * hf + agg).astype(np.float16)
    hd = _up(h, dev)
    z = _buf(n, 0, dev)
    nat.check(nat.lib.gfx_aggregate(problem["handle"], 1, hd.data_ptr(), rp.data_ptr(),
                                    cs.data_ptr(), ct.data_ptr(), n, z.data_ptr(), 0, _stream()))
    torch.cuda.synchronize()
    got = z.cpu().numpy()
    # fma contraction of eps1*h + agg may differ from NumPy's two roundings by one fp16 ulp
    err = np.abs(got.astype(np.float32) - want.astype(np.float32))
    assert err.max() <= 2 ** -10 * max(1.0, np.abs(want.astype(np.float32)).max())
    assert (got != want).mean() < 0.02


@pytest.mark.parametrize("code,impl", [(1, 1), (1, 0), (1, 8), (0, 1), (0, 2), (0, 5)])
def test_mlp_layernorm_residual_layer0(nat, dev, problem, code, impl):
    """K2 (SIMT fp32, split-fp16 tcgen05 for fp32 storage -- the GFX_F32 default --, SIMT fp16-storage,
    general tcgen05, lean tcgen05 + TMA) against the oracle's h1."""
    keep = problem["keep32" if code == 1 else "keep16"]
    tdt = torch.float32 if code == 1 else torch.float16
    n = keep["h0"].shape[0]
    z, h = _up(keep["z0"], dev).to(tdt), _up(keep["h0"], dev).to(tdt)
    out = _buf(n, code, dev)
    nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], 0, z.data_ptr(), h.data_ptr(),
                                          n, out.data_ptr(), code, impl, _stream()))
    torch.cuda.synchronize()
    got, want = out.float().cpu().numpy(), keep["h1"]
    err = np.abs(got - want).max()
    scale = np.abs(want).max()
    # fp32: summation order differs from numpy's matmul -> ~1e-5 relative.
    # fp16 storage: hidden activations round to fp16 in both; a 1-ulp flip of
    # a hidden value moves the LayerNorm input by ~1e-3 relative.
    assert err <= (2e-5 if code == 1 else 4e-3) * scale, (err, scale)


@pytest.mark.parametrize("code,impl,out_code", [(1, 1, 1), (1, 0, 1), (1, 8, 0), (0, 1, 0), (0, 2, 0), (0, 2, 1), (0, 0, 0), (0, 0, 1)])
def test_head_l2norm(nat, dev, problem, code, impl, out_code):
    keep = problem["keep32" if code == 1 else "keep16"]
    y = problem["y32" if code == 1 else "y16"]
    tdt = torch.float32 if code == 1 else torch.float16
    n = y.shape[0]
    h = _up(keep["h4"], dev).to(tdt)
    out = _buf(n, out_code, dev)
    nat.check(nat.lib.gfx_head_l2norm(problem["handle"], h.data_ptr(), None, n,
                                      out.data_ptr(), code, out_code, impl, _stream()))
    torch.cuda.synchronize()
    want = y / np.maximum(np.linalg.norm(y.astype(np.float64), axis=1, keepdims=True), 1e-12)
    got = out.float().cpu().numpy()
    tol = 2e-6 if (code == 1 and out_code == 1) else 1.5e-3
    assert np.abs(got - want).max() <= tol
    assert np.abs(np.linalg.norm(got.astype(np.float64), axis=1) - 1).max() <= (
        1e-5 if out_code == 1 else 2e-3)


@pytest.mark.parametrize("n", [1, 127, 129, 128 * 148 * 4 + 128 * 2 + 77, 128 * 148 * 9 + 5])
def test_head_tma_kernel_against_the_general_one(nat, dev, problem, n):
    """The TMA head (impl 0: fp16 in / fp16 out / no row map, gfx_head8.cu) against the general tcgen05
    head (impl 2) beyond one wave: more than four tiles per CTA (every stage buffer reused, both
    barrier parities), partly filled last tile, rows past n untouched, unit norms."""
    g = torch.Generator(device="cpu").manual_seed(n)
    h = (torch.randn(n, 128, generator=g) * 2).to(dev).half()
    want = torch.empty((n, 128), dtype=torch.float16, device=dev)
    got = torch.full((n + 256, 128), 7.0, dtype=torch.float16, device=dev)
    nat.check(nat.lib.gfx_head_l2norm(problem["handle"], h.data_ptr(), None, n, want.data_ptr(), 0, 0, 2, _stream()))
    nat.check(nat.lib.gfx_head_l2norm(problem["handle"], h.data_ptr(), None, n, got.data_ptr(), 0, 0, 0, _stream()))
    torch.cuda.synchronize()
    assert torch.all(got[n:] == 7.0)
    assert (got[:n].float() - want.float()).abs().max().item() <= 1e-3
    assert (got[:n].float().norm(dim=1) - 1).abs().max().item() <= 2e-3


@pytest.mark.parametrize("entry", ["gfx_layer_fused_pair"])
def test_fused_layer_matches_oracle(nat, dev, problem, entry):
    """K1+K2 in one kernel (aggregation warps feed the tcgen05 pipeline through
    shared memory, on CTA pairs sharing the weights) against
    the oracle's h1 given its h0."""
    fused = getattr(nat.lib, entry)
    keep = problem["keep16"]
    rp, cs, ct = problem["csr"]
    n = keep["h0"].shape[0]
    h = _up(keep["h0"], dev).to(torch.float16)
    out = _buf(n, 0, dev)
    nat.check(fused(problem["handle"], 0, h.data_ptr(), rp.data_ptr(),
                    cs.data_ptr(), ct.data_ptr(), n, out.data_ptr(), _stream()))
    torch.cuda.synchronize()
    got, want = out.float().cpu().numpy(), keep["h1"]
    assert np.abs(got - want).max() <= 4e-3 * np.abs(want).max()
    out2 = _buf(n, 0, dev)
    nat.check(fused(problem["handle"], 0, h.data_ptr(), rp.data_ptr(),
                    cs.data_ptr(), ct.data_ptr(), n, out2.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(out, out2)          # deterministic


def test_fused_layers_follow_the_half_precision_chain_of_the_reference(nat, dev, problem):
    """Both fused layer kernels against the oracle restatement of THEIR arithmetic (the reference's
    fp16 path: fp16 message, fp16 sum chain in CSR order, fp16 fused self term, LayerNorm output
    rounded to fp16 before the fp16 residual add; oracle.forward_folded(half_sums=True)), layer by
    layer from the oracle's own inputs.  What may still differ is the fp32 summation order inside
    the tensor-core GEMMs: an occasional hidden activation or LayerNorm output that sits on a
    rounding boundary flips by one fp16 ulp, i.e. the result is within 2 ulp everywhere and equal
    almost everywhere."""
    keep = problem["keep16s"]
    rp, cs, ct = problem["csr"]
    n = keep["h0"].shape[0]
    desc = torch.empty(n, dtype=torch.int32, device=dev)
    nat.check(nat.lib.gfx_row_describe(rp.data_ptr(), cs.data_ptr(), ct.data_ptr(), n,
                                       desc.data_ptr(), _stream()))
    for layer in range(4):
        h = _up(keep[f"h{layer}"], dev).to(torch.float16)
        want = keep[f"h{layer + 1}"]
        outs = []
        for banded in (False, True):
            out = _buf(n, 0, dev)
            if banded:
                nat.check(nat.lib.gfx_layer_fused_banded(
                    problem["handle"], layer, h.data_ptr(), rp.data_ptr(), cs.data_ptr(),
                    ct.data_ptr(), desc.data_ptr(), n, out.data_ptr(), _stream()))
            else:
                nat.check(nat.lib.gfx_layer_fused_pair(
                    problem["handle"], layer, h.data_ptr(), rp.data_ptr(), cs.data_ptr(),
                    ct.data_ptr(), n, out.data_ptr(), _stream()))
            torch.cuda.synchronize()
            got = out.float().cpu().numpy()
            err = np.abs(got - want)
            assert (err <= 2.0 ** -9 * np.maximum(1.0, np.abs(want))).all(), (layer, banded, err.max())
            assert (got != want).mean() < 0.02, (layer, banded, (got != want).mean())
            outs.append(out)
        assert torch.equal(outs[0], outs[1]), layer        # the two kernels: the same bits


@pytest.mark.parametrize("seed,count", [(41, 1), (42, 2), (43, 3), (44, 7), (45, 40), (46, 333)])
def test_fused_pair_layer_ragged_sizes(nat, dev, problem, seed, count):
    """The CTA-pair kernel on node counts that leave the last tile partly empty, an odd number of
    tiles (the second CTA of the last pair has no rows) or fewer tiles than CTAs: every layer
    against K1 + K2 on the same input."""
    import ginfinity_b200 as g
    shard = g.GraphBuilder().build_shard(random_records(seed, count))
    n = shard.node_count
    rp, cs, ct = device_csr(nat, dev, shard.edge_index, shard.edge_types, n)
    rng = np.random.default_rng(seed)
    h = _up((rng.standard_normal((n, 128)) * 2).astype(np.float16), dev)
    for layer in range(4):
        z = _buf(n, 0, dev)
        want = _buf(n, 0, dev)
        got = torch.full((n + 64, 128), 7.0, dtype=torch.float16, device=dev)   # guard rows
        nat.check(nat.lib.gfx_aggregate(problem["handle"], layer, h.data_ptr(), rp.data_ptr(),
                                        cs.data_ptr(), ct.data_ptr(), n, z.data_ptr(), 0, _stream()))
        nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], layer, z.data_ptr(), h.data_ptr(),
                                              n, want.data_ptr(), 0, 5, _stream()))
        nat.check(nat.lib.gfx_layer_fused_pair(problem["handle"], layer, h.data_ptr(), rp.data_ptr(),
                                               cs.data_ptr(), ct.data_ptr(), n, got.data_ptr(),
                                               _stream()))
        torch.cuda.synchronize()
        assert torch.all(got[n:] == 7.0)                       # nothing written past the last row
        diff = (got[:n].float() - want.float()).abs().max().item()
        assert diff <= 4e-3 * max(1.0, want.float().abs().max().item()), (layer, n, diff)


def _describe_rows(rp, cs, ct):
    return O.describe_rows(rp, cs, ct)     # oracle/gine_oracle.py: the restatement gfx_row_describe is checked against


def _device_describe(nat, dev, rp, cs, ct, n):
    desc = torch.empty(n, dtype=torch.int32, device=dev)
    nat.check(nat.lib.gfx_row_describe(rp.data_ptr(), cs.data_ptr(), ct.data_ptr(), n,
                                       desc.data_ptr(), _stream()))
    return desc


def _banded_vs_pair(nat, dev, problem, rp, cs, ct, n, seed, layers=(0, 1, 2, 3)):
    rng = np.random.default_rng(seed)
    h = _up((rng.standard_normal((n, 128)) * 2).astype(np.float16), dev)
    desc = _device_describe(nat, dev, rp, cs, ct, n)
    for layer in layers:
        want = _buf(n, 0, dev)
        got = torch.full((n + 64, 128), 7.0, dtype=torch.float16, device=dev)   # guard rows
        nat.check(nat.lib.gfx_layer_fused_pair(problem["handle"], layer, h.data_ptr(), rp.data_ptr(),
                                               cs.data_ptr(), ct.data_ptr(), n, want.data_ptr(),
                                               _stream()))
        nat.check(nat.lib.gfx_layer_fused_banded(problem["handle"], layer, h.data_ptr(), rp.data_ptr(),
                                                 cs.data_ptr(), ct.data_ptr(), desc.data_ptr(), n,
                                                 got.data_ptr(), _stream()))
        torch.cuda.synchronize()
        assert torch.all(got[n:] == 7.0)                       # nothing written past the last row
        assert torch.equal(got[:n], want), (layer, n, (got[:n].float() - want.float()).abs().max().item())
    return desc


@pytest.mark.parametrize("seed,count", [(51, 1), (52, 3), (53, 40), (54, 333)])
def test_row_descriptors_and_banded_layer_full_molecules(nat, dev, problem, seed, count):
    """Full-molecule graphs: every row is banded (no GENERIC rows), descriptors equal the NumPy
    restatement bit for bit, and the banded fused layer equals the pair kernel BIT FOR BIT (same
    messages, same summation order) -- including odd tile counts and partly empty last tiles."""
    import ginfinity_b200 as g
    shard = g.GraphBuilder().build_shard(random_records(seed, count))
    n = shard.node_count
    rp, cs, ct = device_csr(nat, dev, shard.edge_index, shard.edge_types, n)
    desc = _banded_vs_pair(nat, dev, problem, rp, cs, ct, n, seed)
    want = _describe_rows(rp.cpu().numpy(), cs.cpu().numpy(), ct.cpu().numpy())
    got = desc.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, want)
    assert not (got & 0x80000000).any()


def test_banded_layer_generic_rows_sliced_windows(nat, dev, problem):
    """Windowed records with context nodes: remapped indices, partners without backbone -- many
    rows are GENERIC and go through the CSR fallback; results still equal the pair kernel's."""
    import ginfinity_b200 as g
    recs = [g.RNA(r.identifier, r.sequence, r.structure, start=r.length // 4, end=r.length // 4 + r.length // 3)
            for r in random_records(61, 60) if r.length >= 40]
    shard = g.GraphBuilder(keep_paired_neighbours=True, context_hops=2).build_shard(recs)
    n = shard.node_count
    rp, cs, ct = device_csr(nat, dev, shard.edge_index, shard.edge_types, n)
    desc = _banded_vs_pair(nat, dev, problem, rp, cs, ct, n, 61, layers=(0, 3))
    got = desc.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, _describe_rows(rp.cpu().numpy(), cs.cpu().numpy(), ct.cpu().numpy()))


def test_banded_layer_arbitrary_graph(nat, dev, problem):
    """A graph that is nothing like an RNA (random sources, duplicate edges, self loops, hubs, all
    ten edge types, isolated nodes): mostly GENERIC rows, a few that happen to look banded."""
    rng = np.random.default_rng(62)
    n, e = 1000, 4000
    dst = rng.integers(0, n, e).astype(np.int32)
    dst[:200] = 7                                               # a hub
    src = rng.integers(0, n, e).astype(np.int32)
    src[200:260] = dst[200:260]                                 # self loops
    typ = rng.integers(0, 10, e).astype(np.uint8)
    # some rows that ARE banded, appended in the canonical order
    extra = []
    for i in (300, 301, 500):
        extra += [(i - 1, i, 0), (i + 1, i, 1), (i + 40, i, 2), (i - 2, i, 4), (i + 2, i, 5)]
    keep = ~np.isin(dst, [300, 301, 500])
    src = np.concatenate([src[keep], np.array([a for a, _, _ in extra], np.int32)])
    dst = np.concatenate([dst[keep], np.array([b for _, b, _ in extra], np.int32)])
    typ = np.concatenate([typ[keep], np.array([c for _, _, c in extra], np.uint8)])
    rp, cs, ct = device_csr(nat, dev, np.stack([src, dst]), typ, n)
    desc = _banded_vs_pair(nat, dev, problem, rp, cs, ct, n, 62, layers=(1,))
    got = desc.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, _describe_rows(rp.cpu().numpy(), cs.cpu().numpy(), ct.cpu().numpy()))
    assert (got[[300, 301, 500]] & 0x3f == 0x37).all() and (got & 0x80000000).sum() > 500


def _edge_describe(nat, dev, edge_index, edge_types, n, base=0):
    """(descriptors, needs_csr flag, status word, workspace) of gfx_edge_describe."""
    ei, et = _up(np.ascontiguousarray(edge_index), dev), _up(np.ascontiguousarray(edge_types), dev)
    e = int(et.shape[0])
    desc = torch.full((n,), -7, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    need = nat.lib.gfx_edge_describe_workspace_bytes(n)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    nat.check(nat.lib.gfx_edge_describe(ei[0].data_ptr() if e else None, ei[1].data_ptr() if e else None,
                                        et.data_ptr() if e else None, n, e, base, desc.data_ptr(),
                                        status.data_ptr(), ws.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    return desc, int(ws[:4].view(torch.int32).item()), int(status.item()), ws, (ei, et)


def test_row_descriptors_from_the_edge_list(nat, dev, problem):
    """gfx_edge_describe (no CSR) against gfx_row_describe on the CSR of the same edges, bit for
    bit: full molecules (all banded, needs_csr = 0), windows with context nodes and an arbitrary
    graph (GENERIC rows, needs_csr = 1), banded rows whose edges appear in another ORDER (the
    summation order would differ: GENERIC), duplicates, an edge that leaves the chunk (dropped
    and reported), a graph without edges; gfx_csr_build_if builds exactly when the flag says so;
    gfx_encode_described computes the bits of gfx_encode(fused = 3)."""
    import ginfinity_b200 as g

    def check(edge_index, edge_types, n, expect_flag=None):
        rp, cs, ct = device_csr(nat, dev, edge_index, edge_types, n)
        want = _device_describe(nat, dev, rp, cs, ct, n).cpu().numpy().view(np.uint32)
        desc, flag, status, ws, (ei, et) = _edge_describe(nat, dev, edge_index, edge_types, n)
        got = desc.cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want)
        assert flag == int(bool((want & 0x80000000).any())) and status == 0
        if expect_flag is not None:
            assert flag == expect_flag
        # the gated build leaves poisoned arrays alone when nothing is GENERIC, else equals K0
        e = int(et.shape[0])
        rp2 = torch.full((n + 1,), -5, dtype=torch.int32, device=dev)
        cs2 = torch.full((max(e, 1),), -5, dtype=torch.int32, device=dev)
        ct2 = torch.full((max(e, 1),), 99, dtype=torch.uint8, device=dev)
        need = nat.lib.gfx_csr_workspace_bytes(n, e)
        cws = torch.empty(need, dtype=torch.uint8, device=dev)
        nat.check(nat.lib.gfx_csr_build_if(ei[0].data_ptr() if e else None, ei[1].data_ptr() if e else None,
                                           et.data_ptr() if e else None, n, e, 0, rp2.data_ptr(),
                                           cs2.data_ptr(), ct2.data_ptr(), ws.data_ptr(),
                                           cws.data_ptr(), need, _stream()))
        torch.cuda.synchronize()
        if flag:
            assert torch.equal(rp2, rp) and torch.equal(cs2[:e], cs[:e]) and torch.equal(ct2[:e], ct[:e])
        else:
            assert bool((rp2 == -5).all()) and bool((cs2 == -5).all())
        return desc, flag, (rp2, cs2, ct2)

    full = g.GraphBuilder().build_shard(random_records(81, 60))
    desc, flag, csr = check(full.edge_index, full.edge_types, full.node_count, expect_flag=0)
    # the described forward == the forward that classifies the CSR rows itself
    x = _up(full.node_features, dev)
    n = full.node_count
    rp, cs, ct = device_csr(nat, dev, full.edge_index, full.edge_types, n)
    need = nat.lib.gfx_encode_workspace_bytes(n, 0)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    a = torch.empty((n, 128), dtype=torch.float16, device=dev)
    b = torch.empty((n, 128), dtype=torch.float16, device=dev)
    nat.check(nat.lib.gfx_encode(problem["handle"], x.data_ptr(), rp.data_ptr(), cs.data_ptr(),
                                 ct.data_ptr(), None, n, a.data_ptr(), 0, 0, 0, 3, ws.data_ptr(), need,
                                 _stream()))
    nat.check(nat.lib.gfx_encode_described(problem["handle"], x.data_ptr(), desc.data_ptr(),
                                           csr[0].data_ptr(), csr[1].data_ptr(), csr[2].data_ptr(), n,
                                           b.data_ptr(), 0, ws.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    assert torch.equal(a, b)

    recs = [g.RNA(r.identifier, r.sequence, r.structure, start=r.length // 4, end=r.length // 4 + r.length // 3)
            for r in random_records(82, 40) if r.length >= 40]
    win = g.GraphBuilder(keep_paired_neighbours=True, context_hops=2).build_shard(recs)
    check(win.edge_index, win.edge_types, win.node_count)

    rng = np.random.default_rng(83)
    n, e = 700, 2500
    src, dst = rng.integers(0, n, e).astype(np.int32), rng.integers(0, n, e).astype(np.int32)
    typ = rng.integers(0, 10, e).astype(np.uint8)
    keep = ~np.isin(dst, [300, 301, 400, 401, 402])
    extra = []
    for i in (300, 301):                                   # banded, canonical order
        extra += [(i - 1, i, 0), (i + 1, i, 1), (i + 40, i, 3), (i - 2, i, 4), (i + 2, i, 5)]
    extra += [(401, 400, 1), (399, 400, 0)]                # banded edges in the wrong order
    extra += [(400, 401, 0), (400, 401, 0)]                # a duplicate
    extra += [(401, 402, 0), (403, 402, 1), (404, 402, 5), (400, 402, 4)]   # skip-2 edges swapped
    src = np.concatenate([src[keep], np.array([a for a, _, _ in extra], np.int32)])
    dst = np.concatenate([dst[keep], np.array([b for _, b, _ in extra], np.int32)])
    typ = np.concatenate([typ[keep], np.array([c for _, _, c in extra], np.uint8)])
    desc, flag, _ = check(np.stack([src, dst]), typ, n, expect_flag=1)
    got = desc.cpu().numpy().view(np.uint32)
    assert (got[[300, 301]] & 0x3f == 0x3f).all() and (got[[400, 401, 402]] == 0x80000000).all()

    check(np.zeros((2, 0), np.int32), np.zeros(0, np.uint8), 5, expect_flag=0)      # no edges at all

    # an edge into another chunk: ignored by the descriptors, reported in the status word
    bad_index = full.edge_index.copy()
    bad_index[0, 7] = full.node_count + 3
    desc2, flag2, status2, _, _ = _edge_describe(nat, dev, bad_index, full.edge_types, full.node_count)
    assert status2 == 16 and flag2 == 0


def test_banded_fp32_aggregate_equals_the_csr_kernel(nat, dev, problem):
    """gfx_aggregate_banded (fp32 storage: K1 from row descriptors, a register window over runs
    of consecutive rows) against gfx_aggregate on the CSR of the same edges, bit for bit: full
    molecules of ragged lengths (runs that start and end inside molecules, a last run shorter
    than 32 rows, partners in other runs), every layer's table; the same shard with one row's
    edges reordered (GENERIC: the device flag sends the chunk to the CSR kernel); tiny chunks;
    gfx_encode_described_f32 == gfx_encode(GFX_F32)."""
    import ginfinity_b200 as g

    def both(edge_index, edge_types, n, h, layer, expect_flag):
        rp, cs, ct = device_csr(nat, dev, edge_index, edge_types, n)
        want = torch.full((n, 128), 7.0, dtype=torch.float32, device=dev)
        nat.check(nat.lib.gfx_aggregate(problem["handle"], layer, h.data_ptr(), rp.data_ptr(),
                                        cs.data_ptr(), ct.data_ptr(), n, want.data_ptr(), 1, _stream()))
        desc, flag, status, ws, (ei, et) = _edge_describe(nat, dev, edge_index, edge_types, n)
        assert flag == expect_flag and status == 0
        got = torch.full((n + 1, 128), -7.0, dtype=torch.float32, device=dev)   # one guard row
        nat.check(nat.lib.gfx_aggregate_banded(problem["handle"], layer, h.data_ptr(), desc.data_ptr(),
                                               ws.data_ptr(), rp.data_ptr(), cs.data_ptr(),
                                               ct.data_ptr(), n, got.data_ptr(), 1, _stream()))
        torch.cuda.synchronize()
        assert torch.equal(got[:n].view(torch.int32), want.view(torch.int32))
        assert bool((got[n] == -7.0).all())
        return desc, ws, (rp, cs, ct)

    full = g.GraphBuilder().build_shard(random_records(91, 90))
    n = full.node_count
    gen = torch.Generator(device="cpu").manual_seed(5)
    h = (torch.randn(n, 128, generator=gen) * 2).to(dev)
    for layer in range(4):
        desc, ws, csr = both(full.edge_index, full.edge_types, n, h, layer, 0)
    # the whole forward from descriptors == the forward on the CSR
    x = _up(full.node_features, dev)
    need = nat.lib.gfx_encode_workspace_bytes(n, 1)
    ews = torch.empty(need, dtype=torch.uint8, device=dev)
    a = torch.empty((n, 128), dtype=torch.float32, device=dev)
    b = torch.empty((n, 128), dtype=torch.float32, device=dev)
    nat.check(nat.lib.gfx_encode(problem["handle"], x.data_ptr(), csr[0].data_ptr(), csr[1].data_ptr(),
                                 csr[2].data_ptr(), None, n, a.data_ptr(), 1, 1, 0, 0, ews.data_ptr(),
                                 need, _stream()))
    nat.check(nat.lib.gfx_encode_described_f32(problem["handle"], x.data_ptr(), desc.data_ptr(),
                                               ws.data_ptr(), None, None, None, n, b.data_ptr(), 1,
                                               ews.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))

    # one row's backbone edges swapped in the edge list: GENERIC, the CSR kernel does the chunk
    ei, et = full.edge_index.copy(), full.edge_types.copy()
    into = np.flatnonzero(ei[1] == 40)
    first, second = into[0], into[1]
    ei[:, [first, second]] = ei[:, [second, first]]
    et[[first, second]] = et[[second, first]]
    both(ei, et, n, h, 1, 1)

    for tiny in (1, 2, 3, 5, 31, 32, 33):                   # chunks shorter than the window / a run
        one = g.GraphBuilder().build_shard([g.RNA("t", ("ACGU" * 9)[:tiny], "." * tiny)])
        hh = (torch.randn(tiny, 128, generator=gen) * 2).to(dev)
        both(one.edge_index, one.edge_types, tiny, hh, 2, 0)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 200, 64 * 3 + 1])
def test_tile_edges(nat, dev, problem, n):
    """Ragged sizes around the 128-row tile / 64-row block boundaries: all
    dense paths agree with SIMT on the first n rows."""
    keep = problem["keep16"]
    z, h = _up(keep["z0"][:n], dev).half(), _up(keep["h0"][:n], dev).half()
    outs = []
    for impl in (1, 2, 5):
        o = _buf(n, 0, dev)
        nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], 0, z.data_ptr(), h.data_ptr(),
                                              n, o.data_ptr(), 0, impl, _stream()))
        outs.append(o)
    torch.cuda.synchronize()
    for o in outs[1:]:
        assert (o.float() - outs[0].float()).abs().max().item() <= 4e-3 * float(np.abs(keep["h1"]).max())


@pytest.mark.parametrize("n", [128 * 3 + 5, 128 * 148 * 5 + 128 * 3 + 17])
def test_mlp_lean_kernel_many_tiles(nat, dev, problem, n):
    """The lean K2 (impl 5) against the general tcgen05 kernel (impl 2) beyond one wave: several
    tiles per CTA (every stage buffer reused, both barrier parities), a partly filled last tile;
    rows past n stay untouched."""
    g = torch.Generator(device="cpu").manual_seed(n)
    z = (torch.randn(n, 128, generator=g) * 3).to(dev).half()
    h = (torch.randn(n, 128, generator=g) * 2).to(dev).half()
    outs = []
    for impl in (2, 5):
        o = torch.full((n + 256, 128), 7.0, dtype=torch.float16, device=dev)
        for layer in (0, 1):
            nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], layer, z.data_ptr(), h.data_ptr(),
                                                  n, o.data_ptr(), 0, impl, _stream()))
        outs.append(o)
    torch.cuda.synchronize()
    assert torch.all(outs[1][n:] == 7.0)
    assert torch.isfinite(outs[1][:n].float()).all()
    diff = (outs[0][:n].float() - outs[1][:n].float()).abs().max().item()
    assert diff <= 4e-3 * max(1.0, outs[0][:n].float().abs().max().item()), (n, diff)


@pytest.mark.parametrize("n", [1, 127, 129, 128 * 3 + 5, 128 * 148 * 2 + 128 + 17])
def test_split_tensor_core_kernels_for_fp32_storage(nat, dev, problem, n):
    """full_precision on the tensor cores (gfx_split9.cu: every fp32 operand as fp16 hi + lo, three
    MMAs per product) against the CUDA-core fp32 kernels on the same inputs: ragged sizes, odd tile
    counts (rank 1 of the last pair idle), several tiles per CTA pair, rows past n untouched, the
    core-row map of the head.  The split is good to 2^-22 per operand: the two paths agree to
    fp32 summation-order noise."""
    g = torch.Generator(device="cpu").manual_seed(n)
    z = (torch.randn(n, 128, generator=g) * 6).to(dev)
    h = (torch.randn(n, 128, generator=g) * 3).to(dev)
    for layer in (0, 3):
        want = torch.empty((n, 128), dtype=torch.float32, device=dev)
        got = torch.full((n + 256, 128), 7.0, dtype=torch.float32, device=dev)
        nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], layer, z.data_ptr(), h.data_ptr(), n,
                                              want.data_ptr(), 1, 1, _stream()))
        nat.check(nat.lib.gfx_mlp_ln_residual(problem["handle"], layer, z.data_ptr(), h.data_ptr(), n,
                                              got.data_ptr(), 1, 8, _stream()))
        torch.cuda.synchronize()
        assert torch.all(got[n:] == 7.0)
        assert (got[:n] - want).abs().max().item() <= 2e-5 * max(1.0, want.abs().max().item()), layer
    # head with a core-row map that drops every third row
    keep = torch.arange(n, device=dev) % 3 != 0
    out_row = torch.where(keep, torch.cumsum(keep.int(), 0) - 1, torch.full((n,), -1, device=dev)).int()
    rows = int(keep.sum().item())
    for out_code, tdt in ((1, torch.float32), (0, torch.float16)):
        want = torch.full((rows + 8, 128), 7.0, dtype=tdt, device=dev)
        got = torch.full((rows + 8, 128), 7.0, dtype=tdt, device=dev)
        nat.check(nat.lib.gfx_head_l2norm(problem["handle"], h.data_ptr(), out_row.data_ptr(), n,
                                          want.data_ptr(), 1, out_code, 1, _stream()))
        nat.check(nat.lib.gfx_head_l2norm(problem["handle"], h.data_ptr(), out_row.data_ptr(), n,
                                          got.data_ptr(), 1, out_code, 8, _stream()))
        torch.cuda.synchronize()
        assert torch.all(got[rows:] == 7.0)
        tol = 2e-6 if out_code == 1 else 1e-3
        if rows:
            assert (got[:rows].float() - want[:rows].float()).abs().max().item() <= tol, out_code


@pytest.mark.parametrize("code,impl,fused", [(1, 1, 0), (1, 0, 0), (0, 1, 0), (0, 2, 0), (0, 5, 0), (0, 5, 2), (0, 5, 3)])
def test_whole_forward(nat, dev, problem, code, impl, fused):
    """gfx_encode (all stages chained on device) against the oracle."""
    x = _up(problem["shard"].node_features, dev)
    rp, cs, ct = problem["csr"]
    n = x.shape[0]
    out = torch.empty((n, 128), dtype=torch.float32, device=dev)
    need = nat.lib.gfx_encode_workspace_bytes(n, code)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    nat.check(nat.lib.gfx_encode(problem["handle"], x.data_ptr(), rp.data_ptr(),
                                 cs.data_ptr(), ct.data_ptr(), None, n, out.data_ptr(),
                                 code, 1, impl, fused, ws.data_ptr(), need, _stream()))
    torch.cuda.synchronize()
    y = problem["y32" if code == 1 else "y16"]
    want = y / np.maximum(np.linalg.norm(y.astype(np.float64), axis=1, keepdims=True), 1e-12)
    got = out.cpu().numpy()
    if code == 1:
        assert np.abs(got - want).max() <= 2e-5
    else:
        # against the fp16-storage oracle, and the north-star bar against fp32
        assert np.abs(got - want).max() <= 3e-3
        y32 = problem["y32"]
        ref = y32 / np.linalg.norm(y32.astype(np.float64), axis=1, keepdims=True)
        cos = (got.astype(np.float64) * ref).sum(1) / np.linalg.norm(got.astype(np.float64), axis=1)
        assert cos.min() >= 0.999

