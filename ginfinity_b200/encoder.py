"""`Ginfinity`: the reference's encoder facade over libgfx.so.

Mirrors src/ginfinity/api.py (reference): `Ginfinity.load`, `encode`,
`encode_many`, `encode_graph`, `encode_graphs`, `graph_spec`,
`embedding_dimension`, `info`, `device`, `full_precision`, with the same
keyword arguments, argument checks, exception types and message fragments
(api.py:64-230), so the reference's tests for this path read the same.

What runs underneath is different.  `_run_graph_shard` in the reference
(api.py:232-260) converts indices to int64, materialises one-hot edge
attributes, runs ~40 eager torch ops per microbatch, normalises in float64
on the host and splits rows in a Python loop.  Here the shard's compact
arrays (float32 features, int32 edge index, uint8 edge types) go to the
device as they are; microbatch boundaries are computed on the device
(gfx_pack_microbatches); consecutive microbatches are grouped into device
chunks; per chunk a destination CSR is built (gfx_csr_build) and the
forward runs as hand-written sm_100a kernels (gfx_encode) ending in the
L2-normalise + cast + core-row compaction epilogue; one device->host copy
per chunk lands in a pinned buffer that the returned per-record arrays are
row-range views of.

Deviations from the reference, all deliberate:
  * only CUDA devices are accepted (no CPU path by mandate);
  * the CUDA path is deterministic (CSR segmented sums, no atomics in
    floating point), so `allow_nondeterministic_cuda` is accepted but not
    required (reference: api.py:71-74);
  * microbatch boundaries do not change any output bit (graphs never
    interact), so chunks of several microbatches are launched together; a
    chunk holds at most CHUNK_MICROBATCHES x max_batch_nodes nodes, so
    lowering `max_batch_nodes` still lowers device memory in proportion
    (reference docs/OPERATIONS.md:25-27);
  * `encode_graphs(..., out=table)` writes into a caller-owned
    [core_count, 128] table (ideally page-locked, see `pinned_table`) and
    returns row-range views of it: a caller that keeps every result pays
    the page-locking cost once, not per call.
"""
from __future__ import annotations

import os

import json
from pathlib import Path
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as nat
from .graph import (Graph, GraphBuilder, GraphCompatibilityError, GraphShard,
                    GraphSpec)
from .weights import (BUNDLED_CONFIG, EncoderConfig, FoldedWeights,
                      ModelIntegrityError, default_model_dir, fold,
                      load_checkpoint, parameter_count)

DEFAULT_CHUNK_NODES = 1 << 20
# device-resident shards have no copy pipeline to keep fine-grained: larger chunks amortise the
# fill and drain of the persistent layer kernel (measured: 2^20 -> 675, 2^21 -> 699 M nt/s with
# the pair kernel; 2^21 -> 708, 2^22 -> 740, 2^23 -> 739 with the banded kernel)
RESIDENT_CHUNK_NODES = 1 << 22
# a chunk never holds more than this many microbatches' worth of nodes (16 x the default 60,000
# is just under 2^20): device scratch scales with max_batch_nodes when the caller lowers it
CHUNK_MICROBATCHES = 16
RESIDENT_CHUNK_MICROBATCHES = 64
GFX_GRAPH_BAD_EDGE = 16            # include/gfx.h


def _embedding_dtype(value) -> np.dtype:
    try:
        dtype = np.dtype(value)
    except TypeError as exc:
        raise ValueError(f"unsupported embedding dtype {value!r}") from exc
    if dtype.kind != "f":
        raise ValueError(f"embedding dtype must be floating-point, got {dtype}")
    return dtype


def default_alignment_parameters(model_dir=None) -> dict:
    """Scoring parameters for the separate SW aligner (api.py:47-50)."""
    root = Path(model_dir) if model_dir is not None else default_model_dir()
    if root is None:
        raise ModelIntegrityError("no model directory has been staged")
    try:
        data = json.loads((root / "alignment.json").read_text())
    except (OSError, json.JSONDecodeError) as exc:
        raise ModelIntegrityError(
            f"cannot read model metadata {root / 'alignment.json'}: {exc}") from exc
    return dict(data["scoring_parameters"])


def _check_architecture(cfg: EncoderConfig) -> None:
    """The kernels implement ONE architecture: h + LayerNorm(...) residual layers
    (_model.py:68-71 with cfg.residual), 7 node features (struct_feature "A",
    positional), hidden = out_dim = 128.  A checkpoint whose config says otherwise
    passes the reference's own checks and would be computed WRONGLY here, so it is
    refused (the reference honours the flags, _model.py:52-60)."""
    problems = []
    if not cfg.residual:
        problems.append("residual=False")
    if cfg.struct_feature != "A" or not cfg.positional:
        problems.append(f"struct_feature={cfg.struct_feature!r}, positional={cfg.positional}")
    if cfg.hidden != 128 or cfg.out_dim != 128:
        problems.append(f"hidden={cfg.hidden}, out_dim={cfg.out_dim}")
    if problems:
        raise ModelIntegrityError(
            "unsupported encoder architecture for the sm_100a kernels: " + "; ".join(problems))


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _as_host_table(out, dtype: np.dtype) -> torch.Tensor:
    """`encode_graphs(out=...)`: a CPU torch view of a caller-owned table."""
    t = torch.from_numpy(out) if isinstance(out, np.ndarray) else out
    if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
        raise ValueError("`out` must be a NumPy array or a CPU torch tensor")
    want = torch.float16 if dtype == np.float16 else torch.float32
    if t.dtype != want or t.dim() != 2 or t.shape[1] != 128 or not t.is_contiguous():
        raise ValueError(f"`out` must be a C-contiguous [rows, 128] table of {dtype}")
    return t


class DeviceShard:
    """A GraphShard's numeric arrays resident in HBM (same dtypes and
    layout as graph.py:261-275; strings stay on the host)."""

    def __init__(self, node_features, edge_index, edge_types, node_ptr,
                 edge_ptr, node_roles, *, max_nodes_per_record: int,
                 max_edges_per_record: int, core_count: int, spec: GraphSpec,
                 core_ptr_host: Optional[np.ndarray] = None):
        self.node_features = node_features
        self.edge_index = edge_index
        self.edge_types = edge_types
        self.node_ptr = node_ptr
        self.edge_ptr = edge_ptr
        self.node_roles = node_roles           # None when every node is core
        self.record_count = int(node_ptr.shape[0]) - 1
        self.node_count = int(node_features.shape[0])
        self.edge_count = int(edge_types.shape[0])
        self.max_nodes_per_record = int(max_nodes_per_record)
        self.max_edges_per_record = int(max_edges_per_record)
        self.core_count = int(core_count)
        self.spec = spec
        self.core_ptr_host = core_ptr_host
        # set once the shard's edges are known to stay inside their chunks (shards from the
        # device builder are; others are checked by the first encode_device_shard)
        self.edges_checked = False

    @property
    def device(self):
        return self.node_features.device

    @classmethod
    def from_shard(cls, shard: GraphShard, device, *, non_blocking=True):
        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(
                device, non_blocking=non_blocking)

        all_core = shard.all_core
        counts = np.diff(shard.node_ptr)
        ecounts = np.diff(shard.edge_ptr)
        if all_core:
            core_ptr, core_count = shard.node_ptr, shard.node_count
        else:
            core_ptr = np.zeros(shard.record_count + 1, np.int64)
            np.cumsum(shard.core_count_array(), out=core_ptr[1:])
            core_count = int(core_ptr[-1])
        return cls(up(shard.node_features), up(shard.edge_index),
                   up(shard.edge_types), up(shard.node_ptr),
                   up(shard.edge_ptr),
                   None if all_core else up(shard.node_roles),
                   max_nodes_per_record=int(counts.max()),
                   max_edges_per_record=int(ecounts.max()),
                   core_count=core_count, spec=shard.spec,
                   core_ptr_host=core_ptr)


class _Scratch:
    """Named device buffers that only ever grow (no allocation in steady state)."""

    def __init__(self, device):
        self.device = device
        self._buf: dict = {}

    def get(self, name: str, nbytes: int) -> torch.Tensor:
        have = self._buf.get(name)
        if have is None or have.numel() < nbytes:
            grow = max(int(nbytes), 1024)
            grow = (grow + grow // 8 + 255) & ~255      # viewable as any dtype
            have = torch.empty(grow, dtype=torch.uint8, device=self.device)
            self._buf[name] = have
        return have


class Ginfinity:
    """Loaded GINFINITY encoder ready for repeated inference on one GPU."""

    def __init__(self, weights: FoldedWeights, metadata: dict, device: str,
                 graph_spec: GraphSpec, *, full_precision: bool):
        _check_architecture(weights.cfg)
        self._weights = weights
        self._metadata = metadata
        self._graph_spec = graph_spec
        self.device = device
        self.full_precision = bool(full_precision)
        self._torch_device = torch.device(device)
        if self._torch_device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        with torch.cuda.device(self._torch_device):
            self._handle = nat.model_create(weights)
        self._scratch = _Scratch(self._torch_device)
        # dense-stage implementation: 0 auto (tcgen05 for fp16), 1 SIMT
        self.impl = nat.IMPL_AUTO
        # layer kernels: 3 = fused layer on CTA pairs with banded producers, 2 = fused layer on CTA
        # pairs with CSR-walking producers (bit-identical to 3; gfx_encode falls back where a
        # kernel does not apply), 0 = K1 + K2.  The default is FIXED (3, with 2 for shards that
        # hold context nodes): every process, rank and run computes with the same kernels, so an
        # input encodes to the same bits fleet-wide (K1 + K2 agree with the fused forms only to
        # fp16 rounding, 2e-3).  GFX_FUSED=0|2|3 pins one form.
        self.fused = 0 if full_precision else int(os.environ.get("GFX_FUSED", "3"))
        self.chunk_nodes = DEFAULT_CHUNK_NODES
        self.resident_chunk_nodes = RESIDENT_CHUNK_NODES
        self.device_builder = True       # encode_many builds full-molecule graphs on the GPU
        # banded layer kernel: row descriptors from the edge list, CSR only for GENERIC rows
        # (False: every chunk through the CSR arrays, the path the tests compare against)
        self.describe_from_edges = True
        self.last_microbatch_bounds: Optional[np.ndarray] = None

    def __del__(self):
        handle, self._handle = getattr(self, "_handle", None), None
        if handle:
            try:
                nat.model_destroy(handle)
            except Exception:
                pass

    # -- construction ------------------------------------------------------
    @staticmethod
    def _check_device(device: str) -> None:
        if not isinstance(device, str) or not device.startswith("cuda"):
            if device == "cpu":
                raise ValueError(
                    "device must be a CUDA device: this build has no CPU path")
            raise ValueError("device must be 'cpu' or a CUDA device")
        if not torch.cuda.is_available():
            raise ValueError("CUDA was requested but is unavailable")

    @classmethod
    def load(cls, device: str = "cuda", *,
             allow_nondeterministic_cuda: bool = False,
             model_dir=None, full_precision: bool = False) -> "Ginfinity":
        """Verify and load a checkpoint directory (api.py:64-114).

        `allow_nondeterministic_cuda` is accepted for signature
        compatibility; this CUDA path is deterministic and does not need it.
        """
        cls._check_device(device)
        root = Path(model_dir) if model_dir is not None else default_model_dir()
        if root is None:
            raise ModelIntegrityError(
                "missing checkpoint: no model_dir given and none staged; run "
                "`python -m ginfinity_b200.stage_model <dir with encoder.pt>`")
        state, cfg, spec, metadata = load_checkpoint(root)
        return cls(fold(state, cfg), metadata, device, spec,
                   full_precision=full_precision)

    @classmethod
    def from_state(cls, state, cfg: EncoderConfig = BUNDLED_CONFIG,
                   device: str = "cuda", *, full_precision: bool = False
                   ) -> "Ginfinity":
        """Build an encoder from an in-memory state dict (tests, benchmarks
        with random-init weights)."""
        cls._check_device(device)
        spec = GraphSpec.from_encoder_config(cfg)
        metadata = {"format_version": 1, "package": "ginfinity_b200",
                    "parameter_count": parameter_count(state),
                    "embedding_dimension": cfg.out_dim,
                    "graph_spec": spec.to_dict(),
                    "graph_spec_sha256": spec.sha256,
                    "checkpoint_sha256": None}
        return cls(fold(state, cfg), metadata, device, spec,
                   full_precision=full_precision)

    # -- properties (api.py:116-126) ---------------------------------------
    @property
    def embedding_dimension(self) -> int:
        return self._weights.cfg.out_dim

    @property
    def graph_spec(self) -> GraphSpec:
        return self._graph_spec

    def info(self) -> dict:
        return json.loads(json.dumps(self._metadata))

    # -- record-level API (api.py:128-178) -----------------------------------
    def encode(self, record, *, keep_paired_neighbours: bool = False,
               context_hops: int = 1, embedding_dtype=np.float16) -> np.ndarray:
        return self.encode_many(
            [record], keep_paired_neighbours=keep_paired_neighbours,
            context_hops=context_hops, embedding_dtype=embedding_dtype)[0]

    def encode_many(self, records: Sequence, *, max_batch_nodes: int = 60_000,
                    max_batch_edges: int = 300_000,
                    keep_paired_neighbours: bool = False, context_hops: int = 1,
                    embedding_dtype=np.float16) -> list:
        records = list(records)
        if not records:
            return []
        if context_hops < 1:                       # GraphBuilder.__init__ (graph.py:476-477)
            raise ValueError("context_hops must be >= 1")
        from . import device_builder
        if self.device_builder and device_builder.supports(self._graph_spec, records):
            if device_builder.any_sliced(records):
                # windowed records: selection + induced subgraphs on the GPU (K7)
                return self._encode_sliced_records(
                    records, int(max_batch_nodes), int(max_batch_edges),
                    bool(keep_paired_neighbours), int(context_hops),
                    _embedding_dtype(embedding_dtype))
            # full-molecule records: graphs are built on the GPU (2 B/nt over PCIe
            # instead of 69 B/nt) group by group, the host preparing group g+1
            # while the device encodes group g and copies out group g-1
            return self._encode_records(records, int(max_batch_nodes), int(max_batch_edges),
                                        _embedding_dtype(embedding_dtype))
        shard = GraphBuilder(
            self._graph_spec, keep_paired_neighbours=keep_paired_neighbours,
            context_hops=context_hops).build_shard(records)
        return self.encode_graphs(shard, max_batch_nodes=max_batch_nodes,
                                  max_batch_edges=max_batch_edges,
                                  embedding_dtype=embedding_dtype)

    def encode_graph(self, graph: Graph, *, embedding_dtype=np.float16
                     ) -> np.ndarray:
        return self.encode_graphs([graph], embedding_dtype=embedding_dtype)[0]

    def _encode_chunk(self, *, src: int, dst: int, typ: int, n: int, e: int, node_base: int, x: int,
                      out_row: Optional[int], out: int, act: int, out_code: int,
                      status: torch.Tensor, stream: int, banded: bool) -> None:
        """One chunk on the current torch stream (`stream` is its raw handle; the arguments are
        device addresses): graph preparation + gfx_encode with the layer kernel of __init__.

        Full-molecule shards of the fp16 model (`banded`): row descriptors straight from the
        edge list (gfx_edge_describe) and a CSR build that runs only if some row is GENERIC
        (gfx_csr_build_if, decided on the device) -- graphs in the reference builder's edge
        order never need the CSR.  Shards with context nodes (whose remapped rows the banded
        kernel would take through its slow GENERIC loop) use the pair kernel, which computes
        the same bits, so a record encodes to the same values alone, in a batch, and next to
        windowed records; K1 + K2 (`GFX_FUSED=0`, full_precision) use the plain CSR."""
        lib = nat.lib
        mode = int(self.fused)
        if mode == 3 and not banded:
            mode = 2
        row_ptr = self._scratch.get("row_ptr", 4 * (n + 1))
        col_src = self._scratch.get("col_src", 4 * max(e, 1))
        col_type = self._scratch.get("col_type", max(e, 1))
        csr_ws_bytes = lib.gfx_csr_workspace_bytes(n, e)
        csr_ws = self._scratch.get("csr_ws", csr_ws_bytes)
        enc_ws_bytes = lib.gfx_encode_workspace_bytes(n, act)
        enc_ws = self._scratch.get("enc_ws", enc_ws_bytes)
        described = (banded and out_row is None and self.describe_from_edges and n <= 1 << 25
                     and (mode == 3 if act == nat.GFX_F16 else self.impl == nat.IMPL_AUTO))
        if described:
            desc = self._scratch.get("desc", 4 * n)
            dws_bytes = lib.gfx_edge_describe_workspace_bytes(n)
            dws = self._scratch.get("desc_ws", dws_bytes)     # its first word: the needs-CSR flag
            nat.check(lib.gfx_edge_describe(src, dst, typ, n, e, node_base, desc.data_ptr(),
                                            status.data_ptr(), dws.data_ptr(), dws_bytes, stream))
            nat.check(lib.gfx_csr_build_if(src, dst, typ, n, e, node_base, row_ptr.data_ptr(),
                                           col_src.data_ptr(), col_type.data_ptr(), dws.data_ptr(),
                                           csr_ws.data_ptr(), csr_ws_bytes, stream))
            if act == nat.GFX_F16:
                nat.check(lib.gfx_encode_described(
                    self._handle, x, desc.data_ptr(), row_ptr.data_ptr(), col_src.data_ptr(),
                    col_type.data_ptr(), n, out, out_code, enc_ws.data_ptr(), enc_ws_bytes, stream))
            else:       # full_precision: K1 from the descriptors, K2 / K3 as split-fp16 GEMMs
                nat.check(lib.gfx_encode_described_f32(
                    self._handle, x, desc.data_ptr(), dws.data_ptr(), row_ptr.data_ptr(),
                    col_src.data_ptr(), col_type.data_ptr(), n, out, out_code, enc_ws.data_ptr(),
                    enc_ws_bytes, stream))
            return
        nat.check(lib.gfx_csr_build_checked(src, dst, typ, n, e, node_base, row_ptr.data_ptr(),
                                            col_src.data_ptr(), col_type.data_ptr(),
                                            status.data_ptr(), csr_ws.data_ptr(), csr_ws_bytes, stream))
        nat.check(lib.gfx_encode(self._handle, x, row_ptr.data_ptr(), col_src.data_ptr(),
                                 col_type.data_ptr(), out_row, n, out, act, out_code, self.impl, mode,
                                 enc_ws.data_ptr(), enc_ws_bytes, stream))

    # -- shard-level API (api.py:180-230) ------------------------------------
    def _check_request(self, spec, max_nodes_per_record, max_edges_per_record,
                       max_batch_nodes, max_batch_edges, embedding_dtype):
        if spec.sha256 != self._graph_spec.sha256:
            raise GraphCompatibilityError(
                "graphs were built with a specification incompatible with "
                "this encoder")
        if max_batch_nodes <= 0 or max_batch_edges <= 0:
            raise ValueError("batch node and edge limits must be positive")
        dtype = _embedding_dtype(embedding_dtype)
        if max_nodes_per_record > max_batch_nodes:
            raise ValueError("max_batch_nodes is smaller than the longest graph")
        if max_edges_per_record > max_batch_edges:
            raise ValueError("max_batch_edges is smaller than the largest graph")
        return dtype

    def encode_graphs(self, graphs, *, max_batch_nodes: int = 60_000,
                      max_batch_edges: int = 300_000,
                      embedding_dtype=np.float16, out=None) -> list:
        """Encode prebuilt graphs; one (core_count_i, 128) array per record,
        in input order.

        `out` (extension; the reference always allocates): a caller-owned
        C-contiguous [total core nodes, 128] table of `embedding_dtype`
        (float16 or float32; NumPy array or CPU torch tensor, ideally
        page-locked: `Ginfinity.pinned_table`).  The embeddings are written
        into it and the returned per-record arrays are row-range views of it,
        so keeping results costs no allocation inside the call."""
        if isinstance(graphs, GraphShard):
            shard = graphs
        else:
            graph_list = list(graphs)
            if not graph_list:
                return []
            shard = GraphShard.from_graphs(graph_list)
        # all argument errors are raised before any device work (api.py:196-210)
        counts = np.diff(shard.node_ptr)
        ecounts = np.diff(shard.edge_ptr)
        dtype = self._check_request(shard.spec, int(counts.max()),
                                    int(ecounts.max()), max_batch_nodes,
                                    max_batch_edges, embedding_dtype)
        out_code = nat.GFX_F16 if dtype == np.float16 else nat.GFX_F32
        host = None
        if out is not None:
            if dtype.itemsize > 4:
                raise ValueError("`out` tables must be float16 or float32")
            host = _as_host_table(out, dtype)
        with torch.cuda.device(self._torch_device), torch.inference_mode():
            table, core_ptr, rows = self._encode_streaming(
                shard, int(max_batch_nodes), int(max_batch_edges), out_code,
                presplit=(dtype.itemsize <= 4), host=host)
        if table.dtype != dtype:
            return split_rows(table.astype(dtype), core_ptr)
        return rows

    @staticmethod
    def pinned_table(rows: int, dtype=np.float16) -> np.ndarray:
        """A page-locked [rows, 128] table for `encode_graphs(..., out=)`.
        Page-locking costs ~0.6 s per GiB (measured, profiles/r01_b_pcie.json):
        allocate once and reuse, or keep a ring of them."""
        tdtype = torch.float16 if np.dtype(dtype) == np.float16 else torch.float32
        t = torch.empty((int(rows), 128), dtype=tdtype, pin_memory=True)
        return t.numpy()

    # -- host shard -> host embeddings, copies overlapped with compute -----------
    def _plan(self, node_ptr_d, edge_ptr_d, B, max_batch_nodes, max_batch_edges,
              stream) -> np.ndarray:  # `stream`: raw handle of the CURRENT torch stream
        """K4 on the device, then one small read-back: rows of (record stop,
        node offset, edge offset) per microbatch boundary."""
        dev = self._torch_device
        next_stop = torch.empty(B, dtype=torch.int64, device=dev)
        bounds = torch.empty(B + 2, dtype=torch.int64, device=dev)
        nat.check(nat.lib.gfx_pack_microbatches(
            node_ptr_d.data_ptr(), edge_ptr_d.data_ptr(), B, max_batch_nodes,
            max_batch_edges, next_stop.data_ptr(), bounds.data_ptr(),
            bounds[B + 1:].data_ptr(), stream))
        stops = bounds[:B + 1].clamp_(0, B)     # the tail past n_bounds is unset
        packed = torch.stack((stops, node_ptr_d[stops], edge_ptr_d[stops]))
        count = int(bounds[B + 1].item())
        plan = packed[:, :count].cpu().numpy()
        self.last_microbatch_bounds = plan[0].copy()
        return plan

    def _chunk_limit(self, max_batch_nodes: int, resident: bool = False) -> int:
        """Nodes per device chunk: the encoder's chunk size, but never more than
        CHUNK_MICROBATCHES microbatches' worth, so that lowering `max_batch_nodes`
        (the reference's memory knob, docs/OPERATIONS.md:25-27) lowers device
        scratch in proportion."""
        if resident:
            return min(max(self.chunk_nodes, self.resident_chunk_nodes),
                       RESIDENT_CHUNK_MICROBATCHES * int(max_batch_nodes))
        return min(self.chunk_nodes, CHUNK_MICROBATCHES * int(max_batch_nodes))

    def _chunks(self, plan: np.ndarray, limit: int, ramp: bool = False) -> list:
        """Group consecutive microbatches into device chunks of at most
        `limit` nodes (always at least one microbatch).  `ramp` (the streaming
        path): the first chunks hold 1/8, 1/4 and 1/2 of `limit`, so the
        device->host copies -- the bottleneck of an end-to-end call, which
        nothing overlaps before the first chunk is encoded -- start after an
        eighth of a chunk's copy-in and compute instead of a whole one."""
        node_at, count = plan[1], plan.shape[1]
        out, start = [], 0
        shift = 3 if ramp else 0
        while start < count - 1:
            cap = limit >> shift
            shift = max(0, shift - 1)
            stop = start + 1
            while (stop < count - 1 and
                   node_at[stop + 1] - node_at[start] <= cap):
                stop += 1
            out.append((start, stop))
            start = stop
        return out

    def _new_status(self) -> torch.Tensor:
        """Device int32 that the CSR builds of one encode OR their complaints into."""
        return torch.zeros(1, dtype=torch.int32, device=self._torch_device)

    @staticmethod
    def _raise_on_status(value: int) -> None:
        if value & GFX_GRAPH_BAD_EDGE:
            from .graph import GraphValidationError
            raise GraphValidationError("edge index outside shard node range")

    def _encode_streaming(self, shard: GraphShard, max_batch_nodes: int,
                          max_batch_edges: int, out_code: int, presplit=True, host=None):
        """Three-stream pipeline over chunks: while chunk c runs on the compute
        stream, chunk c+1's arrays are copied in and chunk c-1's embeddings
        are copied out into one pinned [core_count, 128] table."""
        dev = self._torch_device
        lib = nat.lib
        B, N = shard.record_count, shard.node_count
        act = nat.GFX_F32 if self.full_precision else nat.GFX_F16
        tdtype = torch.float16 if out_code == nat.GFX_F16 else torch.float32
        esize = 2 if out_code == nat.GFX_F16 else 4
        all_core = shard.all_core
        if all_core:
            core_ptr = shard.node_ptr
        else:
            core_ptr = np.zeros(B + 1, np.int64)
            np.cumsum(shard.core_count_array(), out=core_ptr[1:])
        if host is None:
            host = torch.empty((int(core_ptr[-1]), 128), dtype=tdtype, pin_memory=True)
        elif tuple(host.shape) != (int(core_ptr[-1]), 128):
            raise ValueError(f"`out` must have shape ({int(core_ptr[-1])}, 128), "
                             f"got {tuple(host.shape)}")
        status = self._new_status()
        status_host = torch.empty(1, dtype=torch.int32, pin_memory=True)

        main = torch.cuda.current_stream()
        if not hasattr(self, "_streams"):
            self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        s_in, s_out = self._streams
        as_t = lambda a: torch.from_numpy(a)  # noqa: E731  (zero-copy view)
        node_ptr_d = as_t(shard.node_ptr).to(dev, non_blocking=True)
        edge_ptr_d = as_t(shard.edge_ptr).to(dev, non_blocking=True)
        plan = self._plan(node_ptr_d, edge_ptr_d, B, max_batch_nodes,
                          max_batch_edges, main.cuda_stream)
        chunks = self._chunks(plan, self._chunk_limit(max_batch_nodes), ramp=True)
        rec_at, node_at, edge_at = plan[0], plan[1], plan[2]
        out_row = None
        if not all_core:
            roles_d = as_t(shard.node_roles).to(dev, non_blocking=True)
            out_row = torch.empty(N, dtype=torch.int32, device=dev)
            n_core = torch.empty(1, dtype=torch.int64, device=dev)
            need = lib.gfx_core_rows_workspace_bytes(N)
            ws = self._scratch.get("core", need)
            nat.check(lib.gfx_core_rows(roles_d.data_ptr(), N, out_row.data_ptr(),
                                        n_core.data_ptr(), ws.data_ptr(), need,
                                        main.cuda_stream))
        max_n = max(int(node_at[b] - node_at[a]) for a, b in chunks)
        max_e = max(int(edge_at[b] - edge_at[a]) for a, b in chunks)
        feats = as_t(shard.node_features)
        eidx = as_t(shard.edge_index)
        etyp = as_t(shard.edge_types)
        slots = []
        for k in range(2):
            slots.append(dict(
                x=self._scratch.get(f"in_x{k}", 28 * max_n).view(torch.float32),
                src=self._scratch.get(f"in_src{k}", 4 * max(max_e, 1)).view(torch.int32),
                dst=self._scratch.get(f"in_dst{k}", 4 * max(max_e, 1)).view(torch.int32),
                typ=self._scratch.get(f"in_typ{k}", max(max_e, 1)),
                out=self._scratch.get(f"out{k}", 128 * esize * max_n),
                in_ready=torch.cuda.Event(), in_free=torch.cuda.Event(),
                out_ready=torch.cuda.Event(), out_free=torch.cuda.Event()))
        s_in.wait_stream(main)
        s_out.wait_stream(main)

        def copy_in(c):
            a, b = chunks[c]
            slot = slots[c & 1]
            n0, n1 = int(node_at[a]), int(node_at[b])
            e0, e1 = int(edge_at[a]), int(edge_at[b])
            with torch.cuda.stream(s_in):
                if c >= 2:
                    s_in.wait_event(slot["in_free"])
                slot["x"][:7 * (n1 - n0)].copy_(feats[n0:n1].reshape(-1), non_blocking=True)
                if e1 > e0:
                    slot["src"][:e1 - e0].copy_(eidx[0, e0:e1], non_blocking=True)
                    slot["dst"][:e1 - e0].copy_(eidx[1, e0:e1], non_blocking=True)
                    slot["typ"][:e1 - e0].copy_(etyp[e0:e1], non_blocking=True)
                slot["in_ready"].record(s_in)

        copy_in(0)
        for c, (a, b) in enumerate(chunks):
            slot = slots[c & 1]
            if c + 1 < len(chunks):
                copy_in(c + 1)
            n0, n1 = int(node_at[a]), int(node_at[b])
            e0, e1 = int(edge_at[a]), int(edge_at[b])
            n, e = n1 - n0, e1 - e0
            c0, c1 = int(core_ptr[rec_at[a]]), int(core_ptr[rec_at[b]])
            main.wait_event(slot["in_ready"])
            if c >= 2:
                main.wait_event(slot["out_free"])
            # ranks in out_row are shard-global: bias the base so rank c0 lands on row 0
            out_base = slot["out"].data_ptr() - (0 if out_row is None else c0 * 128 * esize)
            self._encode_chunk(
                src=slot["src"].data_ptr(), dst=slot["dst"].data_ptr(), typ=slot["typ"].data_ptr(),
                n=n, e=e, node_base=n0, x=slot["x"].data_ptr(),
                out_row=None if out_row is None else out_row[n0:].data_ptr(), out=out_base, act=act,
                out_code=out_code, status=status, stream=main.cuda_stream, banded=out_row is None)
            slot["in_free"].record(main)
            slot["out_ready"].record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(slot["out_ready"])
                rows = c1 - c0
                if rows:
                    src = slot["out"][:rows * 128 * esize].view(tdtype).view(rows, 128)
                    host[c0:c1].copy_(src, non_blocking=True)
                slot["out_free"].record(s_out)
        status_host.copy_(status, non_blocking=True)
        main.wait_stream(s_out)
        # the per-record views are built while the device is still working
        table = host.numpy()
        rows = split_rows(table, core_ptr) if presplit else None
        main.synchronize()
        self._raise_on_status(int(status_host.item()))
        return table, core_ptr, rows

    records_group_nodes = 1 << 22      # nucleotides per host-prep / device-build group

    def _encode_records(self, records: list, max_batch_nodes: int, max_batch_edges: int,
                        dtype: np.dtype) -> list:
        """records -> embeddings with the graphs built on the device.

        The node limit is checked before any device work, like the reference
        (api.py:196-210); the edge limit as soon as a group's edge counts exist
        (they come out of the device builder's pairing pass)."""
        from . import device_builder as dbuild
        if max_batch_nodes <= 0 or max_batch_edges <= 0:
            raise ValueError("batch node and edge limits must be positive")
        ids = [r.identifier for r in records]
        if len(set(ids)) != len(ids):
            from .graph import GraphValidationError
            raise GraphValidationError("duplicate identifiers in graph shard")
        B = len(records)
        lengths = np.fromiter(map(len, (r.sequence for r in records)), np.int64, B)
        if int(lengths.max()) > max_batch_nodes:
            raise ValueError("max_batch_nodes is smaller than the longest graph")
        node_ptr = np.zeros(B + 1, np.int64)
        np.cumsum(lengths, out=node_ptr[1:])
        N = int(node_ptr[-1])
        out_code = nat.GFX_F16 if dtype == np.float16 else nat.GFX_F32
        tdtype = torch.float16 if out_code == nat.GFX_F16 else torch.float32
        # groups of whole records: small first (nothing overlaps the first group's host
        # preparation), then doubling up to records_group_nodes nucleotides
        cuts, size = [0], max(1, self.records_group_nodes >> 3)
        while cuts[-1] < B:
            target = node_ptr[cuts[-1]] + size
            nxt = int(np.searchsorted(node_ptr, target, side="right")) - 1
            cuts.append(min(B, max(nxt, cuts[-1] + 1)))
            size = min(2 * size, self.records_group_nodes)
        dev = self._torch_device
        with torch.cuda.device(dev), torch.inference_mode():
            host = torch.empty((N, 128), dtype=tdtype, pin_memory=True)
            main = torch.cuda.current_stream()
            if not hasattr(self, "_streams"):
                self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
            s_build, s_out = self._streams
            s_build.wait_stream(main)
            s_out.wait_stream(main)
            state = dict(out_free=[None, None], turn=0, keep=[], status=self._new_status(),
                         limit=self._chunk_limit(max_batch_nodes))
            bounds = [0]
            table = host.numpy()
            presplit = dtype.itemsize <= 4
            rows = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                with torch.cuda.stream(s_build):
                    ds = dbuild.build_device_shard(records[a:b], dev, self._graph_spec,
                                                   lengths=lengths[a:b])
                    if ds.max_edges_per_record > max_batch_edges:
                        torch.cuda.synchronize()
                        raise ValueError("max_batch_edges is smaller than the largest graph")
                    plan = self._plan(ds.node_ptr, ds.edge_ptr, b - a, max_batch_nodes,
                                      max_batch_edges, s_build.cuda_stream)
                    built = torch.cuda.Event()
                    built.record(s_build)
                bounds.extend((plan[0][1:] + a).tolist())
                main.wait_event(built)
                self._enqueue_resident(ds, plan, host[int(node_ptr[a]):int(node_ptr[b])],
                                       out_code, state)
                if presplit:        # per-record views, made while the device is busy
                    rows.extend(split_rows(table, node_ptr[a:b + 1]))
            self.last_microbatch_bounds = np.asarray(bounds, np.int64)
            main.wait_stream(s_out)
            bad = int(state["status"].item())           # synchronises
            state["keep"].clear()
            self._raise_on_status(bad)
        if table.dtype != dtype:
            return split_rows(table.astype(dtype), node_ptr)
        return rows

    def _encode_sliced_records(self, records: list, max_batch_nodes: int, max_batch_edges: int,
                               keep_paired: bool, hops: int, dtype: np.dtype) -> list:
        """Windowed records -> embeddings of their core nucleotides, with the
        selection (graph.py:599-646) and the induced subgraphs (graph.py:649-695)
        made on the device.  Argument errors are raised before the encode, as in
        the reference (api.py:196-210); the per-record sizes they need come out of
        the selection pass."""
        from . import device_builder as dbuild
        from .graph import GraphValidationError
        if hops < 1:
            raise ValueError("context_hops must be >= 1")
        if max_batch_nodes <= 0 or max_batch_edges <= 0:
            raise ValueError("batch node and edge limits must be positive")
        ids = [r.identifier for r in records]
        if len(set(ids)) != len(ids):
            raise GraphValidationError("duplicate identifiers in graph shard")
        dev = self._torch_device
        out_code = nat.GFX_F16 if dtype == np.float16 else nat.GFX_F32
        with torch.cuda.device(dev), torch.inference_mode():
            ds = dbuild.build_device_shard(records, dev, self._graph_spec,
                                           keep_paired_neighbours=keep_paired,
                                           context_hops=hops)
            self._check_request(ds.spec, ds.max_nodes_per_record, ds.max_edges_per_record,
                                max_batch_nodes, max_batch_edges, dtype)
            out = self.encode_device_shard(ds, max_batch_nodes=max_batch_nodes,
                                           max_batch_edges=max_batch_edges,
                                           out_dtype=out_code, _checked=True)
            host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
            host.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        table = host.numpy()
        if table.dtype != dtype:
            table = table.astype(dtype)
        return split_rows(table, ds.core_ptr_host)

    def _enqueue_resident(self, ds: "DeviceShard", plan: np.ndarray, host: torch.Tensor,
                          out_code: int, state: dict) -> None:
        """Enqueue the forward of a device-resident shard of full molecules on
        the current stream, chunk by chunk; each chunk's embeddings are copied
        into `host` ([nodes, 128], pinned) on the copy-out stream while the
        next chunk runs.  Does not synchronise."""
        lib = nat.lib
        act = nat.GFX_F32 if self.full_precision else nat.GFX_F16
        tdtype = torch.float16 if out_code == nat.GFX_F16 else torch.float32
        esize = 2 if out_code == nat.GFX_F16 else 4
        main = torch.cuda.current_stream()
        s_out = self._streams[1]
        chunks = self._chunks(plan, state["limit"])
        node_at, edge_at = plan[1], plan[2]
        max_n = max(int(node_at[b] - node_at[a]) for a, b in chunks)
        max_e = max(int(edge_at[b] - edge_at[a]) for a, b in chunks)
        outs = [self._scratch.get(f"out{k}", 128 * esize * max_n) for k in range(2)]
        state["keep"].append((ds, outs))
        ei = ds.edge_index
        for a, b in chunks:
            n0, n1 = int(node_at[a]), int(node_at[b])
            e0, e1 = int(edge_at[a]), int(edge_at[b])
            n, e = n1 - n0, e1 - e0
            turn = state["turn"]
            state["turn"] = turn ^ 1
            out = outs[turn]
            if state["out_free"][turn] is not None:
                main.wait_event(state["out_free"][turn])
            self._encode_chunk(
                src=ei[0, e0:].data_ptr() if e else None, dst=ei[1, e0:].data_ptr() if e else None,
                typ=ds.edge_types[e0:].data_ptr() if e else None, n=n, e=e, node_base=n0,
                x=ds.node_features[n0:].data_ptr(), out_row=None, out=out.data_ptr(), act=act,
                out_code=out_code, status=state["status"], stream=main.cuda_stream, banded=True)
            ready = torch.cuda.Event()
            ready.record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ready)
                src = out[:n * 128 * esize].view(tdtype).view(n, 128)
                host[n0:n1].copy_(src, non_blocking=True)
                free = torch.cuda.Event()
                free.record(s_out)
                state["out_free"][turn] = free

    def encode_device_shard(self, ds: DeviceShard, *, max_batch_nodes=60_000,
                            max_batch_edges=300_000, out_dtype=nat.GFX_F16,
                            out: Optional[torch.Tensor] = None,
                            _checked: bool = False) -> torch.Tensor:
        """Device-resident encode: HBM in, HBM out ([core_count, 128] in
        `out_dtype`).  Everything is enqueued on the current stream of the
        encoder's device; the only host synchronisation is the read-back of the
        microbatch boundaries -- and, the FIRST time a shard that did not come
        out of the device builder is encoded, of the edge-range status word
        (a shard whose edges leave their chunk raises GraphValidationError, as
        the reference's GraphShard.slice does; afterwards the shard is known
        good and later calls do not wait)."""
        if not _checked:
            self._check_request(ds.spec, ds.max_nodes_per_record,
                                ds.max_edges_per_record, max_batch_nodes,
                                max_batch_edges, np.float16)
        with torch.cuda.device(self._torch_device):
            return self._encode_device_shard(ds, int(max_batch_nodes), int(max_batch_edges),
                                             out_dtype, out)

    def _encode_device_shard(self, ds, max_batch_nodes, max_batch_edges, out_dtype, out):
        dev = self._torch_device
        stream = torch.cuda.current_stream().cuda_stream
        B, N = ds.record_count, ds.node_count
        # ---- K4: microbatch boundaries on the device ----------------------
        next_stop = torch.empty(B, dtype=torch.int64, device=dev)
        bounds = torch.empty(B + 2, dtype=torch.int64, device=dev)
        nat.check(nat.lib.gfx_pack_microbatches(
            ds.node_ptr.data_ptr(), ds.edge_ptr.data_ptr(), B,
            max_batch_nodes, max_batch_edges, next_stop.data_ptr(),
            bounds.data_ptr(), bounds[B + 1:].data_ptr(), stream))
        stops = bounds[:B + 1].clamp_(0, B)     # the tail past n_bounds is unset
        packed = torch.stack((stops, ds.node_ptr[stops], ds.edge_ptr[stops]))
        count = int(bounds[B + 1].item())
        plan = packed[:, :count].cpu().numpy()
        self.last_microbatch_bounds = plan[0].copy()
        # ---- output and core-row map ---------------------------------------
        tdtype = torch.float16 if out_dtype == nat.GFX_F16 else torch.float32
        if out is None:
            out = torch.empty((ds.core_count, 128), dtype=tdtype, device=dev)
        out_row = None
        if ds.node_roles is not None:
            out_row = torch.empty(N, dtype=torch.int32, device=dev)
            n_core = torch.empty(1, dtype=torch.int64, device=dev)
            need = nat.lib.gfx_core_rows_workspace_bytes(N)
            ws = self._scratch.get("core", need)
            nat.check(nat.lib.gfx_core_rows(
                ds.node_roles.data_ptr(), N, out_row.data_ptr(),
                n_core.data_ptr(), ws.data_ptr(), need, stream))
        # ---- chunks of consecutive microbatches ------------------------------
        act = nat.GFX_F32 if self.full_precision else nat.GFX_F16
        node_at, edge_at = plan[1], plan[2]
        limit = self._chunk_limit(max_batch_nodes, resident=True)
        status = self._new_status()
        start = 0
        while start < count - 1:
            stop = start + 1
            while (stop < count - 1 and
                   node_at[stop + 1] - node_at[start] <= limit):
                stop += 1
            n0, n1 = int(node_at[start]), int(node_at[stop])
            e0, e1 = int(edge_at[start]), int(edge_at[stop])
            self._run_chunk(ds, n0, n1, e0, e1, out_row, out, act, out_dtype,
                            stream, status)
            start = stop
        if not getattr(ds, "edges_checked", False):
            self._raise_on_status(int(status.item()))     # synchronises, once per shard
            ds.edges_checked = True
        return out

    def _run_chunk(self, ds, n0, n1, e0, e1, out_row, out, act, out_dtype,
                   stream, status) -> None:
        n, e = n1 - n0, e1 - e0
        ei = ds.edge_index
        if out_row is None:
            out_base = out[n0:].data_ptr()      # identity map: row i -> n0 + i
            map_ptr = None
        else:
            out_base = out.data_ptr()           # ranks in out_row are global
            map_ptr = out_row[n0:].data_ptr()
        self._encode_chunk(
            src=ei[0, e0:].data_ptr() if e else None, dst=ei[1, e0:].data_ptr() if e else None,
            typ=ds.edge_types[e0:].data_ptr() if e else None, n=n, e=e, node_base=n0,
            x=ds.node_features[n0:].data_ptr(), out_row=map_ptr, out=out_base, act=act,
            out_code=out_dtype, status=status, stream=stream, banded=map_ptr is None)


def _check_unique_ids(records) -> None:
    """GraphShard rejects duplicate identifiers (graph.py:288-289); the device
    builder path keeps that contract."""
    from .graph import GraphValidationError
    seen = set()
    for r in records:
        if r.identifier in seen:
            raise GraphValidationError("duplicate identifiers in graph shard")
        seen.add(r.identifier)


def pin_shard(shard: GraphShard) -> GraphShard:
    """Copy of `shard` whose numeric arrays live in page-locked host memory,
    so `encode_graphs` can feed the device with asynchronous DMA copies."""
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
        view = t.numpy()
        np.copyto(view, a)
        return view

    clone = object.__new__(GraphShard)          # already validated: skip re-validation
    for name in ("identifiers", "sequences", "structures", "spec"):
        object.__setattr__(clone, name, getattr(shard, name))
    for name in ("node_features", "edge_index", "edge_types", "node_ptr",
                 "edge_ptr", "residue_index", "node_roles"):
        object.__setattr__(clone, name, pinned(getattr(shard, name)))
    return clone


def split_rows(table: np.ndarray, row_ptr: np.ndarray) -> list:
    """Per-record row-range views of the [total_core, 128] result
    (replaces the per-record mask loop of api.py:253-259)."""
    edges = row_ptr.tolist()
    return [table[a:b] for a, b in zip(edges[:-1], edges[1:])]
