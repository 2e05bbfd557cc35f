"""GPU tests of the `Ginfinity` facade: the reference's own API tests for this
path (tests/test_api.py, tests/test_graph.py, tests/test_sliced_graphs.py in
the reference) restated against ginfinity_b200, plus parity with the golden
embeddings that oracle/make_golden.py recorded from the reference.

Tolerances (BASELINE.json north_star): per-nucleotide cosine >= 0.999 against
the reference fp32 model; max-abs <= 4e-3 against the reference fp16 model
(whose own distance from its fp32 model is 1.5e-3 on these records).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import gine_oracle as O  # noqa: E402
from helpers import random_records  # noqa: E402


@pytest.fixture(scope="module")
def gb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ginfinity_b200
    return ginfinity_b200


@pytest.fixture(scope="module")
def enc16(gb, parity):
    return gb.Ginfinity.load("cuda:0", model_dir=parity.model_dir)


@pytest.fixture(scope="module")
def enc32(gb, parity):
    return gb.Ginfinity.load("cuda:0", model_dir=parity.model_dir, full_precision=True)


@pytest.fixture(scope="module")
def syn16(gb, synthetic_state):
    return gb.Ginfinity.from_state(synthetic_state, device="cuda:0")


def _cos(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


# ---- parity with the reference's recorded outputs ---------------------------
def test_golden_full_records_fp32_model(enc32, golden_shard, parity):
    got = np.concatenate(enc32.encode_graphs(golden_shard, embedding_dtype=np.float32))
    assert got.shape == (golden_shard.node_count, 128)
    got = got[parity.embeddings["full/rows"]]
    ref = parity.embeddings["full/fp32_model_f32"]
    assert np.abs(got - ref).max() <= 2e-5          # fp32 kernels vs torch fp32
    assert _cos(got, ref).min() >= 0.999999


def test_golden_full_records_fp16_model(enc16, golden_shard, parity):
    got = np.concatenate(enc16.encode_graphs(golden_shard))
    assert got.dtype == np.float16 and got.shape == (golden_shard.node_count, 128)
    got = got[parity.embeddings["full/rows"]]
    ref32 = parity.embeddings["full/fp32_model_f32"]
    ref16 = parity.embeddings["full/fp16_model_f16"].astype(np.float32)
    assert _cos(got, ref32).min() >= 0.999           # north-star bar
    assert np.abs(got.astype(np.float32) - ref16).max() <= 4e-3   # north-star bar
    # and in practice we sit closer to the fp32 model than the reference's
    # own fp16 path does
    assert np.abs(got.astype(np.float32) - ref32).max() <= 2.5e-3


def test_golden_windows(gb, enc16, enc32, golden_meta, parity):
    for k, w in enumerate(golden_meta["windows"]):
        r = w["record"]
        rec = gb.RNA(r[0], r[1], r[2], start=r[3], end=r[4])
        kw = dict(keep_paired_neighbours=w["keep"], context_hops=w["hops"])
        got32 = enc32.encode(rec, embedding_dtype=np.float32, **kw)
        ref32 = parity.embeddings[f"window{k}/fp32_model_f32"]
        assert got32.shape == ref32.shape == (r[4] - r[3], 128)
        assert np.abs(got32 - ref32).max() <= 2e-5
        got16 = enc16.encode(rec, **kw)
        ref16 = parity.embeddings[f"window{k}/fp16_model_f16"].astype(np.float32)
        assert np.abs(got16.astype(np.float32) - ref16).max() <= 4e-3


# ---- reference tests/test_api.py, restated ----------------------------------
def test_bundled_model_loads_and_is_deterministic(gb, enc16):
    record = gb.RNA("rna", "ACGUACGU", "((....))")
    first, second = enc16.encode(record), enc16.encode(record)
    assert first.shape == (8, 128) and first.dtype == np.float16
    np.testing.assert_array_equal(first, second)
    np.testing.assert_allclose(np.linalg.norm(first.astype(np.float64), axis=1), 1.0, atol=1e-3)
    assert enc16.info()["parameter_count"] == 306_436
    assert enc16.embedding_dimension == 128
    assert enc16.graph_spec.sha256 == gb.GraphSpec.bundled().sha256


def test_full_precision_model_is_available(gb, enc32):
    assert enc32.full_precision
    assert enc32.encode(gb.RNA("rna", "ACGU", "....")).dtype == np.float16


def test_embedding_dtype_is_configurable(gb, enc16):
    record = gb.RNA("rna", "ACGU", "....")
    assert enc16.encode(record, embedding_dtype="float32").dtype == np.float32
    out64 = enc16.encode_many([record], embedding_dtype=np.float64)[0]
    assert out64.dtype == np.float64
    np.testing.assert_allclose(np.linalg.norm(out64, axis=1), 1.0, atol=1e-6)
    with pytest.raises(ValueError, match="floating-point"):
        enc16.encode(record, embedding_dtype="int8")


def test_batch_preserves_order_and_rejects_duplicates(gb, enc16):
    first, second = gb.RNA("first", "ACGU", "...."), gb.RNA("second", "GGAA", "(())")
    outputs = enc16.encode_many([first, second])
    assert [v.shape[0] for v in outputs] == [4, 4]
    alone = enc16.encode(second)
    np.testing.assert_array_equal(outputs[1], alone)
    with pytest.raises(ValueError, match="duplicate"):
        enc16.encode_many([first, first])
    assert enc16.encode_many([]) == [] and enc16.encode_graphs([]) == []


def test_cpu_device_is_refused(gb):
    with pytest.raises(ValueError, match="CUDA"):
        gb.Ginfinity.load(device="cpu")
    with pytest.raises(ValueError, match="device"):
        gb.Ginfinity.load(device="tpu")


# ---- reference tests/test_graph.py, restated --------------------------------
def test_saved_staged_encoding_equals_direct_encoding_across_microbatches(gb, enc16, tmp_path):
    records = [gb.RNA("rna-1", "ACGUACGU", "((....))"), gb.RNA("rna-2", "GGAACCUU", "........")]
    direct = enc16.encode_many(records, embedding_dtype=np.float32)
    path = tmp_path / "graphs.safetensors"
    gb.save_graph_shard(gb.GraphBuilder().build_shard(records), path)
    restored = gb.load_graph_shard(path, expected_spec=enc16.graph_spec)
    staged = enc16.encode_graphs(restored, max_batch_nodes=8, max_batch_edges=30,
                                 embedding_dtype=np.float32)
    assert enc16.last_microbatch_bounds.tolist() == [0, 1, 2]
    for a, b in zip(direct, staged):
        np.testing.assert_allclose(b, a, rtol=1e-5, atol=3e-7)   # reference's own bar


def test_encoder_rejects_an_incompatible_graph_specification(gb, enc16):
    other = gb.GraphSpec(struct_feature="B", positional=True, edge_dim=10, extra_edges=("skip2",))
    graph = gb.GraphBuilder(other).build(gb.RNA("rna-1", "ACGUACGU", "((....))"))
    with pytest.raises(gb.GraphCompatibilityError, match="incompatible"):
        enc16.encode_graph(graph)


def test_graph_microbatch_limits_reject_one_oversized_graph(gb, enc16):
    graph = gb.GraphBuilder().build(gb.RNA("rna-1", "ACGUACGU", "((....))"))
    with pytest.raises(ValueError, match="max_batch_edges"):
        enc16.encode_graphs([graph], max_batch_edges=29)
    with pytest.raises(ValueError, match="max_batch_nodes"):
        enc16.encode_graphs([graph], max_batch_nodes=7)
    with pytest.raises(ValueError, match="positive"):
        enc16.encode_graphs([graph], max_batch_nodes=0)


# ---- reference tests/test_sliced_graphs.py, restated -------------------------
_STEM = ("stem", "GGGAAACCCUUUUGGG", "......(((....)))")


def test_encode_returns_only_core_rows_in_sequence_order(gb, enc16):
    rec = gb.RNA(*_STEM, start=9, end=16)
    emb = enc16.encode(rec, keep_paired_neighbours=True, context_hops=3)
    assert emb.shape == (7, 128) and emb.dtype == np.float16
    without = enc16.encode(rec)
    assert not np.allclose(without.astype(np.float32), emb.astype(np.float32), atol=1e-3)


def test_mixed_full_and_sliced_records_in_one_shard(real_state, gb, enc16):
    # reference checkpoint only: the seeded weights expose the open issue in DESIGN.md section 4
    recs = [gb.RNA("a", "ACGUACGU", "((....))"), gb.RNA(*_STEM, start=9, end=16),
            gb.RNA("b", "GGAACCUU", "........")]
    outs = enc16.encode_many(recs, keep_paired_neighbours=True, context_hops=2)
    assert [o.shape[0] for o in outs] == [8, 7, 8]
    for rec, o in zip(recs, outs):
        alone = enc16.encode(rec, keep_paired_neighbours=True, context_hops=2)
        np.testing.assert_array_equal(o, alone)


# ---- larger shards: oracle parity, layout invariance, chunking -----------------
def test_synthetic_shard_matches_oracle_and_is_layout_invariant(gb, syn16, synthetic_state):
    shard = gb.GraphBuilder().build_shard(random_records(31, 400))     # ~80k nodes
    fw = O.fold_state(synthetic_state)
    want = np.concatenate(O.encode_shard(fw, shard, embedding_dtype=np.float32,
                                         half_storage=True))
    syn16.chunk_nodes = 30_000          # several chunks, several microbatches each
    a = np.concatenate(syn16.encode_graphs(shard, max_batch_nodes=9_000,
                                           max_batch_edges=45_000,
                                           embedding_dtype=np.float32))
    bounds_small = syn16.last_microbatch_bounds
    lengths, ecounts = np.diff(shard.node_ptr).tolist(), np.diff(shard.edge_ptr).tolist()
    assert np.array_equal(bounds_small, O.pack_microbatches(lengths, ecounts, 9_000, 45_000))
    syn16.chunk_nodes = 1 << 19
    b = np.concatenate(syn16.encode_graphs(shard, embedding_dtype=np.float32))
    assert np.array_equal(a, b)         # microbatch/chunk layout changes no bit
    assert np.abs(a - want).max() <= 3e-3
    assert _cos(a, want).min() >= 0.9999


def test_fixed_layer_kernel_and_all_forms_agree(gb, syn16, synthetic_state, monkeypatch):
    """The fp16 model's layer runs as one kernel on CTA pairs (banded producers, or producers that
    walk the CSR arrays: same bits) or as K1 + K2 (agrees to fp16 rounding only).  The choice is
    FIXED (banded, pair for shards with context nodes) so that an input encodes to the same bits
    on every board, rank and run.  All forms stay within the fp16-path tolerance of the oracle and
    of each other."""
    shard = gb.GraphBuilder().build_shard(random_records(35, 120))
    monkeypatch.delenv("GFX_FUSED", raising=False)
    fresh = gb.Ginfinity.from_state(synthetic_state, device="cuda:0")
    assert fresh.fused == 3
    auto = np.concatenate(fresh.encode_graphs(shard, embedding_dtype=np.float32))
    assert fresh.fused == 3                                # nothing was timed, nothing changed
    outs = {}
    for mode in (0, 2, 3):
        pinned = gb.Ginfinity.from_state(synthetic_state, device="cuda:0")
        pinned.fused = mode
        outs[mode] = np.concatenate(pinned.encode_graphs(shard, embedding_dtype=np.float32))
    assert np.array_equal(auto, outs[3])
    assert np.array_equal(outs[2], outs[3])                # same messages, same summation order
    assert np.abs(outs[0] - outs[2]).max() <= 2e-3
    fw = O.fold_state(synthetic_state)
    want = np.concatenate(O.encode_shard(fw, shard, embedding_dtype=np.float32, half_storage=True))
    for mode in (0, 2, 3):
        assert np.abs(outs[mode] - want).max() <= 3e-3
        assert _cos(outs[mode], want).min() >= 0.9999
    # windowed records with context nodes: pinned to the banded form or not, same bits as mode 2
    recs = [gb.RNA(r.identifier, r.sequence, r.structure, start=r.length // 4, end=r.length // 2)
            for r in random_records(36, 40)]
    kw = dict(keep_paired_neighbours=True, context_hops=2, embedding_dtype=np.float32)
    win = {}
    for mode in (2, 3):
        pinned = gb.Ginfinity.from_state(synthetic_state, device="cuda:0")
        pinned.fused = mode
        win[mode] = np.concatenate(pinned.encode_many(recs, **kw))
    assert np.array_equal(win[2], win[3])
    full = gb.Ginfinity.from_state(synthetic_state, device="cuda:0", full_precision=True)
    assert full.fused == 0                                 # fp32 model: K1 + K2 (SIMT) only


def test_full_precision_from_row_descriptors_equals_the_csr_path(gb, synthetic_state):
    """full_precision=True: K1 from row descriptors (gfx_encode_described_f32, the default for
    full-molecule shards) gives the bits of K1 on the CSR arrays (describe_from_edges = False),
    over several chunks and microbatches, host path and device-resident path; a shard whose edge
    order is not the reference builder's takes the CSR kernel through the device flag and still
    agrees."""
    from ginfinity_b200.encoder import DeviceShard
    enc = gb.Ginfinity.from_state(synthetic_state, device="cuda:0", full_precision=True)
    shard = gb.GraphBuilder().build_shard(random_records(37, 120))
    limits = dict(max_batch_nodes=3000, max_batch_edges=15_000, embedding_dtype=np.float32)
    keep = enc.chunk_nodes, enc.resident_chunk_nodes
    enc.chunk_nodes = enc.resident_chunk_nodes = 7000
    try:
        assert enc.describe_from_edges
        a = np.concatenate(enc.encode_graphs(shard, **limits))
        ds = DeviceShard.from_shard(shard, "cuda:0")
        c = enc.encode_device_shard(ds, max_batch_nodes=3000, max_batch_edges=15_000,
                                    out_dtype=1).cpu().numpy()
        # the same edges, the first record's edge list reversed: rows of that record are GENERIC
        e1 = int(shard.edge_ptr[1])
        ei, et = shard.edge_index.copy(), shard.edge_types.copy()
        ei[:, :e1] = ei[:, :e1][:, ::-1]
        et[:e1] = et[:e1][::-1]
        other = _clone_shard(gb, shard, edge_index=ei, edge_types=et)
        d = np.concatenate(enc.encode_graphs(other, **limits))
        enc.describe_from_edges = False
        b = np.concatenate(enc.encode_graphs(shard, **limits))
        e = np.concatenate(enc.encode_graphs(other, **limits))
    finally:
        enc.chunk_nodes, enc.resident_chunk_nodes = keep
    assert np.array_equal(a, b) and np.array_equal(a, c)
    assert np.array_equal(d, e)
    n1 = int(shard.node_ptr[1])
    assert np.array_equal(d[n1:], a[n1:]) and np.abs(d[:n1] - a[:n1]).max() < 1e-5


def test_simt_and_tcgen05_paths_agree(gb, syn16):
    from ginfinity_b200 import _native as nat
    shard = gb.GraphBuilder().build_shard(random_records(32, 60))
    syn16.impl = nat.IMPL_UMMA
    a = np.concatenate(syn16.encode_graphs(shard, embedding_dtype=np.float32))
    syn16.impl = nat.IMPL_SIMT
    b = np.concatenate(syn16.encode_graphs(shard, embedding_dtype=np.float32))
    syn16.impl = nat.IMPL_AUTO
    assert np.abs(a - b).max() <= 2e-3


# ---- BASELINE configs[2]: long RNAs, dense long-range pairs, big microbatches -----
def test_long_rna_shard_matches_oracle_across_microbatch_limits(gb, syn16, synthetic_state):
    """1-10 knt records (past RNA's 4096-nt cap, built from duck-typed records
    the way SURVEY 8d C3 prescribes): irregular aggregation with pairs that
    span thousands of rows, and microbatch limits from one graph per batch to
    the whole shard in one."""
    from ginfinity_b200.synthetic import synthetic_records
    recs = synthetic_records(1, 6, lo=1000, hi=10000, log_uniform=True, workers=1)
    shard = gb.GraphBuilder().build_shard(recs)
    longest, most_edges = int(np.diff(shard.node_ptr).max()), int(np.diff(shard.edge_ptr).max())
    assert longest > 4096
    span = np.abs(shard.edge_index[0].astype(np.int64) - shard.edge_index[1])
    assert span.max() > 1000                       # genuinely long-range pairs
    fw = O.fold_state(synthetic_state)
    want = np.concatenate(O.encode_shard(fw, shard, max_batch_nodes=1 << 20,
                                         max_batch_edges=1 << 23,
                                         embedding_dtype=np.float32, half_storage=True))
    outs = []
    for nodes, edges in ((longest, most_edges), (60_000, 300_000), (1 << 20, 1 << 23)):
        outs.append(np.concatenate(syn16.encode_graphs(
            shard, max_batch_nodes=nodes, max_batch_edges=edges, embedding_dtype=np.float32)))
        lengths, ecounts = np.diff(shard.node_ptr).tolist(), np.diff(shard.edge_ptr).tolist()
        assert np.array_equal(syn16.last_microbatch_bounds,
                              O.pack_microbatches(lengths, ecounts, nodes, edges))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[1], outs[2])
    assert np.abs(outs[0] - want).max() <= 3e-3
    assert _cos(outs[0], want).min() >= 0.9999
    assert np.abs(np.linalg.norm(outs[0].astype(np.float64), axis=1) - 1).max() <= 1e-6
    with pytest.raises(ValueError, match="max_batch_nodes"):
        syn16.encode_graphs(shard, max_batch_nodes=longest - 1)


def test_maximum_length_record_and_tiny_records(gb, syn16, synthetic_state):
    """RNA's own limits: one 4096-nt record next to 1-, 2- and 3-nt records
    (0, 2 and 8 edges) in the same shard."""
    rng = np.random.default_rng(5)
    from ginfinity_b200.synthetic import random_structure
    big = "".join(rng.choice(list("ACGU"), 4096))
    recs = [gb.RNA("big", big, random_structure(rng, 4096)), gb.RNA("one", "A", "."),
            gb.RNA("two", "AC", ".."), gb.RNA("three", "GAC", "(.)")]
    shard = gb.GraphBuilder().build_shard(recs)
    assert np.diff(shard.edge_ptr).tolist()[1:] == [0, 2, 8]
    got = syn16.encode_graphs(shard, embedding_dtype=np.float32)
    want = O.encode_shard(O.fold_state(synthetic_state), shard, embedding_dtype=np.float32,
                          half_storage=True)
    assert [g.shape for g in got] == [(4096, 128), (1, 128), (2, 128), (3, 128)]
    for g, w in zip(got, want):
        assert np.abs(g - w).max() <= 3e-3


def test_encode_shard_files_with_prefetch_matches_direct_encoding(gb, syn16, tmp_path):
    """The C4 unit of work: shard files assigned to ranks by node count, the
    next file loaded and pinned while the current one is encoded."""
    from ginfinity_b200.multi_gpu import assign_shards, encode_shard_files
    paths, shards = [], []
    for k in range(4):
        shard = gb.GraphBuilder().build_shard(random_records(40 + k, 30 + 10 * k, prefix=f"f{k}-"))
        path = tmp_path / f"part-{k}.safetensors"
        gb.save_graph_shard(shard, path)
        paths.append(str(path))
        shards.append(shard)
    counts = [s.node_count for s in shards]
    seen = {}
    for rank in range(2):
        seen.update(encode_shard_files(syn16, paths, rank=rank, world_size=2))
        seen_plain = encode_shard_files(syn16, paths, rank=rank, world_size=2, prefetch=False,
                                        node_counts=counts)
        for p, arrays in seen_plain.items():
            assert all(np.array_equal(a, b) for a, b in zip(arrays, seen[p]))
    assert sorted(seen) == sorted(paths)
    assert sorted(sum(assign_shards(counts, 2), [])) == [0, 1, 2, 3]
    for p, shard in zip(paths, shards):
        want = syn16.encode_graphs(shard)
        assert len(want) == len(seen[p])
        assert all(np.array_equal(a, b) for a, b in zip(want, seen[p]))


# ---- round-2 contract additions ------------------------------------------------------------
def _clone_shard(gb, shard, **replace):
    fields = {name: getattr(shard, name) for name in (
        "identifiers", "sequences", "structures", "node_features", "edge_index", "edge_types",
        "node_ptr", "edge_ptr", "spec", "residue_index", "node_roles")}
    fields.update(replace)
    return gb.GraphShard(**fields)


def test_edges_that_leave_their_chunk_are_rejected_not_dereferenced(gb, syn16):
    """A shard that passes construction-time validation (every index in [0, N)) but holds an edge
    into another microbatch: the reference raises GraphValidationError when GraphShard.slice
    re-validates the microbatch (graph.py:328-330, 424-443).  Here the CSR build drops the edge
    (no out-of-range device access) and the encode raises the same error -- on the host path, on
    the device-resident path (first use of the shard), and nothing is poisoned afterwards.
    (Like the reference, which only sees an edge that leaves its MICROBATCH, this path only sees
    an edge that leaves its CHUNK of microbatches; inside one both compute it as given.)"""
    from ginfinity_b200.encoder import DeviceShard
    shard = gb.GraphBuilder().build_shard(random_records(71, 60))
    good = np.concatenate(syn16.encode_graphs(shard, embedding_dtype=np.float32))
    ei = shard.edge_index.copy()
    ei[0, 3] = shard.node_count - 1            # source in the LAST record, destination in the first
    bad = _clone_shard(gb, shard, edge_index=ei)
    limits = dict(max_batch_nodes=2000, max_batch_edges=10_000)     # several microbatches / chunks
    keep = syn16.chunk_nodes, syn16.resident_chunk_nodes
    syn16.chunk_nodes = syn16.resident_chunk_nodes = 4000
    try:
        with pytest.raises(gb.GraphValidationError, match="outside shard node range"):
            syn16.encode_graphs(bad, **limits)
        with pytest.raises(gb.GraphValidationError, match="outside shard node range"):
            syn16.encode_device_shard(DeviceShard.from_shard(bad, "cuda:0"), **limits)
        again = np.concatenate(syn16.encode_graphs(shard, embedding_dtype=np.float32, **limits))
    finally:
        syn16.chunk_nodes, syn16.resident_chunk_nodes = keep
    assert np.array_equal(again, good)


def test_caller_owned_result_table(gb, syn16):
    """encode_graphs(out=table): embeddings land in the caller's (page-locked) table, the returned
    arrays are views of it, the bits are those of the allocating call; wrong tables are refused
    before any device work."""
    shard = gb.GraphBuilder().build_shard(random_records(72, 50))
    want = syn16.encode_graphs(shard)
    table = gb.Ginfinity.pinned_table(shard.node_count)
    assert table.shape == (shard.node_count, 128) and table.dtype == np.float16
    got = syn16.encode_graphs(shard, out=table)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    assert all(np.shares_memory(a, table) for a in got)
    table32 = np.empty((shard.node_count, 128), np.float32)          # pageable memory also works
    got32 = syn16.encode_graphs(shard, embedding_dtype=np.float32, out=table32)
    assert np.shares_memory(got32[0], table32)
    assert np.abs(np.concatenate(got32) - np.concatenate(want).astype(np.float32)).max() <= 1e-3
    with pytest.raises(ValueError, match="out"):
        syn16.encode_graphs(shard, out=np.empty((shard.node_count - 1, 128), np.float16))
    with pytest.raises(ValueError, match="out"):
        syn16.encode_graphs(shard, out=np.empty((shard.node_count, 128), np.float32))
    with pytest.raises(ValueError, match="out"):
        syn16.encode_graphs(shard, embedding_dtype=np.float64,
                            out=np.empty((shard.node_count, 128), np.float64))


def test_lowering_max_batch_nodes_lowers_device_scratch(gb, synthetic_state):
    """The reference's memory knob (docs/OPERATIONS.md:25-27): a chunk holds at most
    CHUNK_MICROBATCHES x max_batch_nodes nodes, so the scratch buffers shrink with it; the bits
    do not change."""
    from ginfinity_b200 import encoder as E
    shard = gb.GraphBuilder().build_shard(random_records(73, 400))       # ~80k nodes
    longest = int(np.diff(shard.node_ptr).max())
    sizes, outs = {}, {}
    for limit in (60_000, max(longest, 500)):
        enc = gb.Ginfinity.from_state(synthetic_state, device="cuda:0")
        outs[limit] = np.concatenate(enc.encode_graphs(
            shard, max_batch_nodes=limit, max_batch_edges=5 * limit + 100))
        sizes[limit] = sum(t.numel() for t in enc._scratch._buf.values())
        assert enc._chunk_limit(limit) == min(enc.chunk_nodes, E.CHUNK_MICROBATCHES * limit)
    small = max(longest, 500)
    assert np.array_equal(outs[60_000], outs[small])
    assert sizes[small] * 4 < sizes[60_000]
