"""Per-nucleotide similarity search over an embedding database (north-star
item 4).  The reference has no counterpart: it only exports scoring
parameters for a separate Smith-Waterman aligner (src/ginfinity/api.py:47-50),
so the contract here is this package's own:

  * database rows and queries are vectors of dimension 128, float16 (what
    `Ginfinity.encode_graphs` returns by default) or float32 (the
    `full_precision=True` output, e.g. `encode_device_shard(out_dtype=GFX_F32)`
    straight from HBM); an index keeps its rows' dtype (`EmbeddingIndex.dtype`)
    and its queries must have the same one.  `metric="cosine"` scores by dot
    product (the encoder's outputs are unit vectors), `metric="l2"` by
    negative squared Euclidean distance;
  * results are ordered by (score descending, database index ascending);
    scores are the sequential fp32 FMA chain over dimensions 0..127 of the
    inputs as given (fp16 or fp32; for L2 the difference is taken in fp32 and
    squared by FMA), so they are reproducible bit for bit on any rank layout.
    A float32 index therefore orders rows that fp16 rounding would make equal;
  * the result is exact for every input.  A tensor-core scan keeps a few
    candidates per database segment, which are rescored exactly; a query is
    certified when the highest tensor-core score the scan dropped, plus a
    margin (2^-14 |q| N_max for cosine, N_max the largest row norm; see
    csrc/gfx_topk.cu), is below its k-th exact score, so no dropped row can
    reach the top k.  Queries that fail are rescored exactly against every
    row on the device in the same call.  A database with one very large-norm
    row, or with many near-duplicates of a query's best rows, pays for that
    fallback; `EmbeddingIndex.last_fallbacks()` counts the queries that took it;
  * float32 rows are scanned as split fp16 (x = hi + lo, three fp16 MMAs per
    product, hi.hi + hi.lo + lo.hi: three times the tensor work of an fp16
    index), with a margin of about 2^-13 |q| N_max.  The index builds the
    [rows, 256] fp16 image hi | lo once and keeps it beside the fp32 rows
    (1 KB per row in all).  A database component above 65504 in magnitude has
    no fp16 hi part and is refused at construction; such a query component is
    accepted and sends that query to the exact fallback;
  * multi-GPU: every rank holds a contiguous row range of the database
    (`EmbeddingIndex.shard`), queries are replicated, each rank takes its
    local top-k on its own GPU (gfx_topk / gfx_topk_f32: tcgen05 GEMM with the
    running top-k fused into the TMEM epilogue), the [Q, k] lists are
    all-gathered with NCCL over NVLink and merged on every rank
    (gfx_topk_merge).

Everything runs through libgfx.so; there is no torch.matmul / topk fallback.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import _native as nat

METRICS = {"cosine": 0, "l2": 1}
MAX_K = 24
DIM = 128


def shard_bounds(num_rows: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced row range [lo, hi) of `rank` (first `num_rows %
    world_size` ranks get one extra row)."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("rank must be in [0, world_size)")
    base, extra = divmod(int(num_rows), world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


DTYPES = (torch.float16, torch.float32)
FP16_MAX = 65504.0


def _as_device_rows(a, device, dtypes, what) -> torch.Tensor:
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a))
    if a.dim() != 2 or a.shape[1] != DIM:
        raise ValueError(f"expected a [rows, {DIM}] array, got {tuple(a.shape)}")
    if a.dtype not in dtypes:
        names = " or ".join(str(d).replace("torch.", "") for d in dtypes)
        raise ValueError(f"{what} must be {names}, got {str(a.dtype).replace('torch.', '')}")
    return a.to(device, non_blocking=True).contiguous()


class EmbeddingIndex:
    """One rank's rows of the embedding database, resident in HBM.

    `database` is a [rows, 128] float16 or float32 array or tensor (a CUDA
    tensor on `device` is used in place, without a copy); the index keeps
    that dtype (`dtype`) and `search` takes queries of the same dtype.  A
    float32 index also keeps the [rows, 256] fp16 split image of its rows
    that its tensor-core scan reads, and refuses a database with a component
    above 65504 in magnitude (one host synchronisation)."""

    def __init__(self, database, *, device="cuda", index_base: int = 0,
                 total_rows: Optional[int] = None):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device: this build has no CPU path")
        self.database = _as_device_rows(database, self.device, DTYPES, "embeddings")
        self.dtype = self.database.dtype
        self.index_base = int(index_base)
        self.total_rows = int(total_rows if total_rows is not None
                              else self.index_base + self.database.shape[0])
        self._ws: Optional[torch.Tensor] = None
        self._image: Optional[torch.Tensor] = None
        if self.dtype == torch.float32 and len(self):
            if not float(self.database.abs().max()) <= FP16_MAX:
                raise ValueError("a float32 database component exceeds 65504 in magnitude, "
                                 "the fp16 range of the split scan (or is NaN)")
            self._image = torch.empty((len(self), 2 * DIM), dtype=torch.float16,
                                      device=self.device)
            with torch.cuda.device(self.device):
                nat.check(nat.lib.gfx_topk_f32_prepare(
                    self.database.data_ptr(), len(self), self._image.data_ptr(),
                    torch.cuda.current_stream().cuda_stream))

    @classmethod
    def shard(cls, database, *, rank: int, world_size: int, device="cuda"):
        """The rows of a host-resident database that belong to `rank`."""
        lo, hi = shard_bounds(database.shape[0], world_size, rank)
        return cls(database[lo:hi], device=device, index_base=lo,
                   total_rows=database.shape[0])

    def __len__(self) -> int:
        return int(self.database.shape[0])

    # -- local search ---------------------------------------------------------
    def search(self, queries, k: int = 10, metric: str = "cosine"
               ) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k of this rank's rows: (scores float32 [Q,k], index int64 [Q,k])
        on the device, indices global (`index_base` added); slots beyond the
        number of rows hold (-inf, -1).  `queries` [Q, 128] must have the
        index's dtype."""
        if metric not in METRICS:
            raise ValueError(f"metric must be one of {sorted(METRICS)}")
        if not 1 <= int(k) <= MAX_K:
            raise ValueError(f"k must be in [1, {MAX_K}]")
        q = _as_device_rows(queries, self.device, (self.dtype,), "queries of this index")
        Q, D = int(q.shape[0]), len(self)
        scores = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        index = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        if Q == 0:
            if self._ws is not None:
                self._ws[:8].zero_()       # no query took the fallback
            return scores, index
        f32 = self.dtype == torch.float32
        with torch.cuda.device(self.device):
            need = (nat.lib.gfx_topk_f32_workspace_bytes if f32
                    else nat.lib.gfx_topk_workspace_bytes)(Q, D, int(k))
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            stream = torch.cuda.current_stream().cuda_stream
            db = self.database.data_ptr() if D else None
            if f32:
                nat.check(nat.lib.gfx_topk_f32(
                    q.data_ptr(), Q, db, self._image.data_ptr() if D else None, D, DIM,
                    int(k), METRICS[metric], self.index_base, scores.data_ptr(),
                    index.data_ptr(), self._ws.data_ptr(), self._ws.numel(), stream))
            else:
                nat.check(nat.lib.gfx_topk(
                    q.data_ptr(), Q, db, D, DIM,
                    int(k), METRICS[metric], self.index_base, scores.data_ptr(),
                    index.data_ptr(), self._ws.data_ptr(), self._ws.numel(), stream))
        return scores, index

    def last_fallbacks(self) -> int:
        """Number of queries of the last `search` on this index that took the
        exact fallback (their candidates could not be certified).  gfx_topk and
        gfx_topk_f32 keep this count as an int64 in the first 8 bytes of its workspace;
        reading it waits for the search to finish."""
        if self._ws is None:
            return 0
        return int(self._ws[:8].view(torch.int64).item())

    # -- sharded search -----------------------------------------------------------
    def search_sharded(self, queries, k: int = 10, metric: str = "cosine", *,
                       group=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Global top-k over all ranks' rows; every rank gets the same result.
        One collective: an all-gather of the [Q, k] score and index lists
        (NCCL over NVLink / NVSwitch), then a k-way merge kernel."""
        import torch.distributed as dist
        scores, index = self.search(queries, k, metric)
        if not (dist.is_available() and dist.is_initialized()):
            return scores, index
        world = dist.get_world_size(group)
        if world == 1:
            return scores, index
        all_scores, all_index = gather_lists(scores, index, world, group)
        return merge_lists(all_scores, all_index)


def gather_lists(scores: torch.Tensor, index: torch.Tensor, world: int, group=None):
    """[Q,k] per rank -> [world, Q, k] on every rank (rank order)."""
    import torch.distributed as dist
    all_scores = torch.empty((world,) + tuple(scores.shape), dtype=scores.dtype,
                             device=scores.device)
    all_index = torch.empty((world,) + tuple(index.shape), dtype=index.dtype,
                            device=index.device)
    # concatenation along dim 0 (the layout both NCCL and gloo accept)
    dist.all_gather_into_tensor(all_scores.view(-1, scores.shape[-1]), scores.contiguous(),
                                group=group)
    dist.all_gather_into_tensor(all_index.view(-1, index.shape[-1]), index.contiguous(),
                                group=group)
    return all_scores, all_index


def merge_lists(all_scores: torch.Tensor, all_index: torch.Tensor):
    """k-way merge of [parts, Q, k] lists (device tensors) by (score desc,
    index asc); entries with index < 0 are padding."""
    if all_scores.device.type != "cuda":
        raise ValueError("merge_lists runs on the GPU (gfx_topk_merge); got a CPU tensor")
    parts, Q, k = (int(v) for v in all_scores.shape)
    out_s = torch.empty((Q, k), dtype=torch.float32, device=all_scores.device)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=all_scores.device)
    with torch.cuda.device(all_scores.device):
        nat.check(nat.lib.gfx_topk_merge(
            all_scores.contiguous().data_ptr(), all_index.contiguous().data_ptr(),
            parts, Q, k, out_s.data_ptr(), out_i.data_ptr(),
            torch.cuda.current_stream().cuda_stream))
    return out_s, out_i
