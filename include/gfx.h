/*
 * gfx.h -- C ABI of libgfx.so, the B200 (sm_100a) GINFINITY encoder path.
 *
 * The reference (nicoaira/GINFINITY 1.2.1) has no FFI layer: its hot path is
 * the Python method Ginfinity._run_graph_shard (src/ginfinity/api.py:232-260)
 * calling GINEEncoder.forward (src/ginfinity/_model.py:65-72).  The entry
 * points below are what a binding for that path replaces; each one cites the
 * reference lines it stands in for.  INTEGRATION.md shows the ctypes stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary
 *   - every pointer is a DEVICE pointer unless the name ends in _host
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default)
 *   - all work is enqueued on `stream`; no call synchronises the device
 *     except gfx_model_create / gfx_model_destroy
 *   - return 0 on success, a GFX_ERR_* code otherwise; the message for the
 *     calling thread's last failure is gfx_last_error()
 *   - no hidden device allocation after gfx_model_create: scratch space is
 *     passed in, sized by the *_workspace_bytes queries
 *   - dtype codes: GFX_F16 = IEEE half storage with fp32 accumulation
 *     (reference default, api.py:111-112), GFX_F32 = fp32 storage
 *     (full_precision=True)
 */
#ifndef GFX_H_
#define GFX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GFX_ABI_VERSION 1

enum {
  GFX_OK = 0,
  GFX_ERR_ARGUMENT = 1,
  GFX_ERR_CUDA = 2,
  GFX_ERR_WORKSPACE = 3,
  GFX_ERR_UNSUPPORTED = 4
};

enum { GFX_F16 = 0, GFX_F32 = 1 };

/* which implementation runs the dense stages */
enum {
  GFX_IMPL_AUTO = 0,  /* tcgen05 for GFX_F16, split-fp16 tcgen05 for GFX_F32 */
  GFX_IMPL_SIMT = 1,  /* CUDA-core fp32-accumulate kernels */
  GFX_IMPL_UMMA = 2,  /* general tcgen05.mma / TMEM kernel (GFX_F16 only; cross-check) */
  GFX_IMPL_UMMA_LEAN = 5, /* K2 default: TMA tile I/O + 16 lean epilogue warps, constants as
                             kernel parameters (codes 3, 4, 6, 7 named variants that were
                             measured in round 1 and removed; they are rejected) */
  GFX_IMPL_SPLIT = 8      /* GFX_F32 default for K2 / K3: every fp32 operand as fp16 hi + lo, three
                             tcgen05 MMAs per product on CTA pairs (fp32-grade results: the
                             reference's full_precision path on the tensor cores) */
};

int gfx_abi_version(void);
const char *gfx_last_error(void);

/* ------------------------------------------------------------------------
 * Model.  Folded weights as produced by ginfinity_b200.weights.fold():
 * eval BatchNorm folded into W1/b1 (_model.py:35), edge_lin(one_hot(t))
 * tabulated as table[l][t][:] = W_e[:,t] + b_e (_model.py:33,43 with
 * api.py:243-245), eps1[l] = 1 + eps_l (_model.py:46).
 * Replaces: model.load_state_dict + .to(device) + .half() (api.py:101-112).
 * ------------------------------------------------------------------------ */
typedef struct {
  int32_t hidden;      /* 128 */
  int32_t layers;      /* 4   */
  int32_t out_dim;     /* 128 */
  int32_t feature_dim; /* 7   */
  int32_t edge_dim;    /* 10  */
  const float *w_in_host; /* [hidden, feature_dim] */
  const float *b_in_host; /* [hidden] */
  const float *table_host; /* [layers, edge_dim, hidden] */
  const float *eps1_host;  /* [layers] */
  const float *w1_host;    /* [layers, 2*hidden, hidden]  (BN folded) */
  const float *b1_host;    /* [layers, 2*hidden] */
  const float *w2_host;    /* [layers, hidden, 2*hidden] */
  const float *b2_host;    /* [layers, hidden] */
  const float *ln_g_host;  /* [layers, hidden] */
  const float *ln_b_host;  /* [layers, hidden] */
  const float *wa_host;    /* [hidden, hidden]   head.0 */
  const float *ba_host;    /* [hidden] */
  const float *wb_host;    /* [out_dim, hidden]  head.2 */
  const float *bb_host;    /* [out_dim] */
} gfx_folded_weights;

typedef struct gfx_model gfx_model;

int gfx_model_create(const gfx_folded_weights *weights, gfx_model **out);
int gfx_model_destroy(gfx_model *model);

/* ------------------------------------------------------------------------
 * K4  microbatch packing on device.  Replaces the greedy contiguous
 * first-fit loop of encode_graphs (api.py:211-229); bit-identical
 * boundaries.  node_ptr / edge_ptr are the shard's int64 [B+1] arrays
 * (graph.py:271-272).  next_stop is scratch [B].  bounds receives
 * [0, stop_1, ..., B] and n_bounds its length (both device).
 * ------------------------------------------------------------------------ */
int gfx_pack_microbatches(const int64_t *node_ptr, const int64_t *edge_ptr,
                          int64_t num_records, int64_t max_batch_nodes,
                          int64_t max_batch_edges, int64_t *next_stop,
                          int64_t *bounds, int64_t *n_bounds, void *stream);

/* ------------------------------------------------------------------------
 * K0  destination-CSR build.  Replaces the per-layer
 * index_select / index_add_ addressing (_model.py:41-45): edges
 * [edge_begin, edge_begin+E) of a shard's (2,E_total) int32 edge_index are
 * stably sorted by destination.  node_base is subtracted from both
 * endpoints (what GraphShard.slice does on the host, graph.py:424-427).
 * Output: row_ptr int32 [N+1], col_src int32 [E], col_type uint8 [E];
 * bit-identical to numpy.argsort(dst, kind="stable").
 * ------------------------------------------------------------------------ */
size_t gfx_csr_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int gfx_csr_build(const int32_t *edge_src, const int32_t *edge_dst,
                  const uint8_t *edge_type, int64_t num_nodes,
                  int64_t num_edges, int32_t node_base, int32_t *row_ptr,
                  int32_t *col_src, uint8_t *col_type, void *workspace,
                  size_t workspace_bytes, void *stream);
/* The same, reporting edges that leave the chunk.  An edge with an endpoint
 * outside [node_base, node_base + num_nodes) is dropped (it would index past
 * the chunk's arrays) and GFX_GRAPH_BAD_EDGE is OR-ed into *status (device
 * int32, zeroed by the caller; may be shared by all chunks of a shard).  The
 * reference raises GraphValidationError("edge index outside shard node
 * range") for the same shard when GraphShard.slice re-validates the
 * microbatch (graph.py:328-330, 424-443); the encoder raises it after the
 * pass when the status word is set.  gfx_csr_build drops silently. */
enum { GFX_GRAPH_BAD_EDGE = 16 };
int gfx_csr_build_checked(const int32_t *edge_src, const int32_t *edge_dst,
                          const uint8_t *edge_type, int64_t num_nodes,
                          int64_t num_edges, int32_t node_base,
                          int32_t *row_ptr, int32_t *col_src,
                          uint8_t *col_type, int32_t *status, void *workspace,
                          size_t workspace_bytes, void *stream);

/* Row descriptors of the banded fused layer straight from the edge list, and a
 * CSR build that only runs when they say it is needed.  For graphs in the
 * reference builder's edge order (graph.py:494-561) every row is banded and
 * the layer kernel never reads the CSR arrays: gfx_edge_describe (one pass over
 * the edges, one over the nodes) replaces K0 + gfx_row_describe for them.
 *   desc      uint32 [num_nodes], bit-identical to gfx_row_describe on the CSR
 *             of the same edges
 *   status    device int32, OR-ed with GFX_GRAPH_BAD_EDGE like
 *             gfx_csr_build_checked (such edges are ignored)
 *   workspace its first int32 is the needs_csr flag: 1 when some row is GENERIC
 *             (anything but a banded row), else 0.  gfx_csr_build_if takes that
 *             pointer: its kernels return at once when the flag is 0, so no
 *             host synchronisation is needed to decide. */
size_t gfx_edge_describe_workspace_bytes(int64_t num_nodes);
int gfx_edge_describe(const int32_t *edge_src, const int32_t *edge_dst,
                      const uint8_t *edge_type, int64_t num_nodes,
                      int64_t num_edges, int32_t node_base, uint32_t *desc,
                      int32_t *status, void *workspace, size_t workspace_bytes,
                      void *stream);
int gfx_csr_build_if(const int32_t *edge_src, const int32_t *edge_dst,
                     const uint8_t *edge_type, int64_t num_nodes,
                     int64_t num_edges, int32_t node_base, int32_t *row_ptr,
                     int32_t *col_src, uint8_t *col_type,
                     const int32_t *needs_csr, void *workspace,
                     size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * K6  graph construction on the device, for full-molecule records of the
 * bundled graph specification.  Replaces GraphBuilder._build_full,
 * _pair_table and GraphShard.from_graphs (graph.py:494-561, 737-747,
 * 376-412); every output array is bit-identical to the reference's.
 *   sequences / structures: the records' strings concatenated, one ASCII
 *     byte per nucleotide ('A','C','G','U' / '(', ')', '.'), uint8 [N]
 *   node_ptr: int64 [B+1] prefix sums of the record lengths
 *   pos_table: float32 [T,2] (sin, cos) rows tabulated ON THE HOST with NumPy
 *     for every distinct record length (the reference's float32 expression,
 *     graph.py:510-514, is not correctly rounded, so it cannot be recomputed
 *     on the device bit for bit); pos_offset: int64 [B], first table row of
 *     each record
 * Two phases, because the edge total is only known after pairing:
 *   gfx_graph_count  -> edge_ptr int64 [B+1] (edge_ptr[B] = E) and *status
 *   (host reads E and allocates edge_index int32 [2,E], edge_types uint8 [E])
 *   gfx_graph_fill   -> node_features float32 [N,7], edge_index (global node
 *     indices), edge_types, optional residue_index int32 [N] / node_roles
 *     uint8 [N] (may be NULL)
 * Both calls take the same workspace.  *status (device int32) collects
 * GFX_GRAPH_BAD_BASE / UNBALANCED / BAD_STRUCTURE bits.
 * ------------------------------------------------------------------------ */
enum { GFX_GRAPH_BAD_BASE = 1, GFX_GRAPH_UNBALANCED = 2, GFX_GRAPH_BAD_STRUCTURE = 4 };
size_t gfx_graph_workspace_bytes(int64_t num_nodes, int64_t num_records);
int gfx_graph_count(const uint8_t *structures, const int64_t *node_ptr,
                    int64_t num_records, int64_t num_nodes, int skip2,
                    int64_t *edge_ptr, int32_t *status, void *workspace,
                    size_t workspace_bytes, void *stream);
int gfx_graph_fill(const uint8_t *sequences, const uint8_t *structures,
                   const int64_t *node_ptr, const int64_t *edge_ptr,
                   int64_t num_records, int64_t num_nodes, int64_t num_edges,
                   int skip2, const float *pos_table, const int64_t *pos_offset,
                   float *node_features, int32_t *edge_index, uint8_t *edge_types,
                   int32_t *residue_index, uint8_t *node_roles, int32_t *status,
                   void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * K7  windowed ("sliced") records on the device.  Replaces
 * _select_slice_nodes, _extract_slice and GraphShard.from_graphs
 * (graph.py:599-695, 376-412) for the bundled graph specification; every
 * output array is bit-identical to the reference's.
 *   sequences / structures / full_ptr: the FULL molecules, as for K6
 *     (uint8 [NF], int64 [B+1])
 *   win_start / win_end: int32 [B], the core window [start, end) of each
 *     record in full-molecule coordinates; a record without a window is
 *     [0, L) (everything kept, every node core)
 *   keep_paired_neighbours / context_hops: GraphBuilder's arguments
 *     (graph.py:471-476); hop 1 adds the pairing partners of core
 *     nucleotides, hops 2.. the graph neighbours of the previous hop's
 *     additions
 * Two phases, because the sliced totals are only known after selection:
 *   gfx_slice_select -> node_ptr, edge_ptr int64 [B+1] of the SLICED shard
 *   (host reads N = node_ptr[B], E = edge_ptr[B] and allocates the outputs)
 *   gfx_slice_fill   -> node_features float32 [N,7] (rows of the full
 *     molecule's features), edge_index int32 [2,E] (shard-global indices,
 *     full-graph edge order), edge_types, residue_index int32 [N] (position
 *     in the full molecule), node_roles uint8 [N] (0 core, 1 context)
 * pos_table / pos_offset as for K6, tabulated for the FULL lengths.
 * *status additionally collects GFX_GRAPH_BAD_WINDOW.
 * ------------------------------------------------------------------------ */
enum { GFX_GRAPH_BAD_WINDOW = 8 };
size_t gfx_slice_workspace_bytes(int64_t num_full_nodes, int64_t num_records);
int gfx_slice_select(const uint8_t *structures, const int64_t *full_ptr,
                     const int32_t *win_start, const int32_t *win_end,
                     int64_t num_records, int64_t num_full_nodes, int skip2,
                     int keep_paired_neighbours, int context_hops,
                     int64_t *node_ptr, int64_t *edge_ptr, int32_t *status,
                     void *workspace, size_t workspace_bytes, void *stream);
int gfx_slice_fill(const uint8_t *sequences, const uint8_t *structures,
                   const int64_t *full_ptr, const int32_t *win_start,
                   const int32_t *win_end, const int64_t *node_ptr,
                   const int64_t *edge_ptr, int64_t num_records,
                   int64_t num_full_nodes, int64_t num_nodes, int64_t num_edges,
                   int skip2, const float *pos_table, const int64_t *pos_offset,
                   float *node_features, int32_t *edge_index, uint8_t *edge_types,
                   int32_t *residue_index, uint8_t *node_roles, int32_t *status,
                   void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * Core-row map.  Replaces the per-record boolean masks of api.py:253-259:
 * out_row[i] = rank of node i among nodes with node_roles == 0, or -1 for
 * context nodes; n_core receives the number of core nodes (device int64).
 * ------------------------------------------------------------------------ */
size_t gfx_core_rows_workspace_bytes(int64_t num_nodes);
int gfx_core_rows(const uint8_t *node_roles, int64_t num_nodes,
                  int32_t *out_row, int64_t *n_core, void *workspace,
                  size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * Stage kernels (one reference op group each).  h / z buffers are
 * [num_nodes, hidden] row-major in `dtype` storage.
 * ------------------------------------------------------------------------ */

/* h = x W_in^T + b_in            (_model.py:55,67; x is float32 [N,7]) */
int gfx_input_linear(const gfx_model *model, const float *x,
                     int64_t num_nodes, void *h, int dtype, void *stream);

/* K1: z_i = (1+eps_l) h_i + sum_{e: dst=i} relu(h[src_e] + table_l[type_e])
 *                                (_model.py:41-46) */
int gfx_aggregate(const gfx_model *model, int layer, const void *h,
                  const int32_t *row_ptr, const int32_t *col_src,
                  const uint8_t *col_type, int64_t num_nodes, void *z,
                  int dtype, void *stream);

/* K1 for GFX_F32 storage from ROW DESCRIPTORS (gfx_edge_describe) instead of the
 * CSR arrays: when `*needs_csr == 0` (device flag written by gfx_edge_describe:
 * every row of the chunk is one of the reference builder's banded rows,
 * graph.py:494-561) a register-window kernel walks runs of consecutive rows and
 * loads each h row once; otherwise the CSR kernel of gfx_aggregate runs on the
 * arrays gfx_csr_build_if built.  Exactly one of the two does the work, decided
 * on the device; both give the bits of gfx_aggregate.  (_model.py:41-46) */
int gfx_aggregate_banded(const gfx_model *model, int layer, const void *h,
                         const uint32_t *desc, const int32_t *needs_csr,
                         const int32_t *row_ptr, const int32_t *col_src,
                         const uint8_t *col_type, int64_t num_nodes, void *z,
                         int dtype, void *stream);

/* K2: h_out = h + LayerNorm_l(W2 relu(W1' z + b1') + b2)
 *                                (_model.py:34-36, 68-71) */
int gfx_mlp_ln_residual(const gfx_model *model, int layer, const void *z,
                        const void *h, int64_t num_nodes, void *h_out,
                        int dtype, int impl, void *stream);

/* K1+K2 in one kernel (z never leaves the SM) on CTA pairs (tcgen05 cta_group::2: the pair shares
 * the weights, each CTA keeps its tile of h resident as neighbour source,
 * residual and output staging); GFX_F16 only, <= 10 edge types, <= 2^27 nodes */
int gfx_layer_fused_pair(const gfx_model *model, int layer, const void *h,
                         const int32_t *row_ptr, const int32_t *col_src,
                         const uint8_t *col_type, int64_t num_nodes, void *h_out,
                         void *stream);

/* Banded form of the fused layer.  gfx_row_describe classifies every CSR row once per chunk:
 * desc[i] says which of (i-1, type 0) (i+1, type 1) [(partner, type 2|3)] (i-2, type 4)
 * (i+2, type 5) -- the reference builder's edge order for nucleotide i (graph.py:494-561) --
 * the row holds, plus the partner index, or marks the row GENERIC.  gfx_layer_fused_banded
 * computes the same layer as gfx_layer_fused_pair, bit for bit, reading banded rows from a
 * register window over the resident h tile and GENERIC rows from the CSR arrays.
 * GFX_F16 only, >= 6 edge types, <= 2^25 nodes. */
int gfx_row_describe(const int32_t *row_ptr, const int32_t *col_src,
                     const uint8_t *col_type, int64_t num_nodes, uint32_t *desc,
                     void *stream);
int gfx_layer_fused_banded(const gfx_model *model, int layer, const void *h,
                           const int32_t *row_ptr, const int32_t *col_src,
                           const uint8_t *col_type, const uint32_t *desc,
                           int64_t num_nodes, void *h_out, void *stream);

/* K3: y = Wb relu(Wa h + ba) + bb; out[out_row[i]] = y_i / max(|y_i|, 1e-12)
 * cast to out_dtype.  out_row == NULL means identity.
 *                                (_model.py:61-63,72; api.py:250-259) */
int gfx_head_l2norm(const gfx_model *model, const void *h,
                    const int32_t *out_row, int64_t num_nodes, void *out,
                    int dtype, int out_dtype, int impl, void *stream);

/* ------------------------------------------------------------------------
 * Whole forward over one packed chunk of graphs (all stages above in
 * order).  Replaces Ginfinity._run_graph_shard's device work
 * (api.py:236-252).  workspace holds the activation ping-pong buffers.
 * `impl`: GFX_IMPL_* for the dense stages.  `fused` (GFX_F16 only) selects the
 * layer kernel: 0 = K1 + K2 (gfx_aggregate, gfx_mlp_ln_residual),
 * 2 (or 1) = gfx_layer_fused_pair, 3 = gfx_row_describe once +
 * gfx_layer_fused_banded per layer (descriptors live in the z buffer, which the
 * fused forms do not use); a form that does not cover the call (edge types,
 * node count) falls back to the next lower one that does.
 * ------------------------------------------------------------------------ */
size_t gfx_encode_workspace_bytes(int64_t num_nodes, int dtype);
int gfx_encode(const gfx_model *model, const float *x, const int32_t *row_ptr,
               const int32_t *col_src, const uint8_t *col_type,
               const int32_t *out_row, int64_t num_nodes, void *out, int dtype,
               int out_dtype, int impl, int fused, void *workspace,
               size_t workspace_bytes, void *stream);

/* The same forward for the fp16 model with the banded fused layer and row
 * descriptors supplied by the caller (gfx_edge_describe): row_ptr / col_src /
 * col_type are read only for GENERIC rows (gfx_csr_build_if built them iff
 * there are any).  Every node is a core node (no out_row map). */
int gfx_encode_described(const gfx_model *model, const float *x,
                         const uint32_t *desc, const int32_t *row_ptr,
                         const int32_t *col_src, const uint8_t *col_type,
                         int64_t num_nodes, void *out, int out_dtype,
                         void *workspace, size_t workspace_bytes, void *stream);

/* The same for the fp32 model (full_precision, api.py:110-112): K1 per layer by
 * gfx_aggregate_banded (`needs_csr`: the flag gfx_edge_describe wrote; the CSR
 * arrays are read only when it is set), K2 / K3 as in gfx_encode(GFX_F32). */
int gfx_encode_described_f32(const gfx_model *model, const float *x,
                             const uint32_t *desc, const int32_t *needs_csr,
                             const int32_t *row_ptr, const int32_t *col_src,
                             const uint8_t *col_type, int64_t num_nodes,
                             void *out, int out_dtype, void *workspace,
                             size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * K5  similarity search (no reference counterpart; north-star item 4).
 * queries [Q,dim], database [D,dim] are GFX_F16 row-major unit vectors.
 * metric 0 = cosine (dot product), 1 = L2 (ranked by -|q-d|^2).
 * Result order: score descending, database index ascending on ties;
 * out_scores float32 [Q,k], out_index int64 [Q,k] (index + index_base).
 * Scores are the sequential fp32 FMA chain over dimensions 0..127, and the
 * result is exact for every input: a tensor-core scan picks kc candidates per
 * database segment, the candidates are rescored exactly, and each query is
 * certified when the highest tensor-core score the scan dropped, plus a
 * margin of 2^-14 |q| N_max (L2: 2^-14 (2 |q| N_max + N_max^2 + |q|^2);
 * N_max the largest row norm), is below its k-th exact score.  Queries that
 * fail the certificate are rescored exactly against every row, on the
 * device, within the same call.  A database with one very large-norm row, or
 * with many near-duplicates of a query's best rows, pays for that fallback.
 * The first 8 bytes of the workspace hold, after the call, the number of
 * queries that took it (int64).
 *
 * float32 inputs (the encoder's full_precision output): gfx_topk_f32 has the
 * same contract over float32 queries and rows -- scores are the sequential
 * fp32 FMA chain over the fp32 values (L2: the difference in fp32, squared by
 * FMA), same order, padding, certificate-and-fallback and workspace header.
 * Its scan multiplies the split-fp16 images x = hi + lo, hi = fp16(x),
 * lo = fp16(x - hi): three fp16 MMAs per K step (hi.hi + hi.lo + lo.hi), so
 * its margin is 2^-13 |q| N_max + 2^-21 (|q| + N_max) (L2:
 * 2^-13 (2 |q| N_max + N_max^2 + |q|^2) + 2^-20 (|q| + N_max)).
 * gfx_topk_f32_prepare writes the database's [rows, 256] fp16 image hi | lo
 * once (`image`: rows * 512 bytes, 16-byte aligned); every row component
 * must be at most 65504 in magnitude (the fp16 range of hi).  A query
 * component above that is allowed: the query takes the exact fallback.
 * The queries' image is built per call in the workspace.
 * ------------------------------------------------------------------------ */
size_t gfx_topk_workspace_bytes(int64_t num_queries, int64_t num_rows, int k);
int gfx_topk(const void *queries, int64_t num_queries, const void *database,
             int64_t num_rows, int dim, int k, int metric, int64_t index_base,
             float *out_scores, int64_t *out_index, void *workspace,
             size_t workspace_bytes, void *stream);
int gfx_topk_f32_prepare(const float *database, int64_t num_rows, void *image,
                         void *stream);
size_t gfx_topk_f32_workspace_bytes(int64_t num_queries, int64_t num_rows, int k);
int gfx_topk_f32(const float *queries, int64_t num_queries, const float *database,
                 const void *image, int64_t num_rows, int dim, int k, int metric,
                 int64_t index_base, float *out_scores, int64_t *out_index,
                 void *workspace, size_t workspace_bytes, void *stream);

/* k-way merge of `parts` per-query sorted lists (all-gathered from the
 * ranks) into the global top-k: in_* are [parts, Q, k]. */
int gfx_topk_merge(const float *in_scores, const int64_t *in_index, int parts,
                   int64_t num_queries, int k, float *out_scores,
                   int64_t *out_index, void *stream);

/* ------------------------------------------------------------------------
 * K8  local alignment of embedding segments (Smith-Waterman, affine gaps;
 * no reference counterpart: the reference ships parameters for an external
 * aligner, api.py:47-50, and this contract is the library's own).
 * queries [q_rows,128], targets [t_rows,128]: GFX_F16 row-major tables (may
 * be the same).  pairs int64 [P,4]: (q_start, q_len, t_start, t_len), rows
 * q_start .. q_start+q_len-1 of queries against t_start .. of targets, each
 * length 0..4096 and inside its table.  For query row i and target row j of a
 * pair, every operation fp32 round-to-nearest, in this order:
 *   S(i,j) = q_i . t_j     tcgen05.mma: fp16 inputs, fp32 accumulation
 *   s      = S(i,j) - offset
 *   E(i,j) = max(H(i,j-1) - gap_open, E(i,j-1) - gap_extend)   gap in the query
 *   F(i,j) = max(H(i-1,j) - gap_open, F(i-1,j) - gap_extend)   gap in the target
 *   H(i,j) = max(0, H(i-1,j-1) + s, E(i,j), F(i,j))
 *   H(-1,.) = H(.,-1) = 0,  E(.,-1) = F(-1,.) = -inf
 * Ties: a positive H takes its start from the first of diagonal, E, F that
 * attains it; a diagonal step from H = 0 starts at (i,j), otherwise the start
 * is inherited; E and F prefer opening to extending; the end cell is the
 * largest H, then the smallest i, then the smallest j.
 * Output: out_score float32 [P] (the largest H); out_coords int32 [P,4] =
 * (query_begin, query_end, target_begin, target_end), half-open, relative to
 * the segments.  No positive cell (zero-length segments included): score 0,
 * coordinates -1.  A pair outside these limits gets score NaN and -1 (the
 * kernel reads nothing for it); callers validate.
 * Accuracy: |S - exact| <= 2^-14 |q_i| |t_j| (kAlignRel in gfx_align.cu), so the
 * score is within min(q_len, t_len) 2^-14 max|q| max|t| of the float64
 * optimum, plus (q_len + t_len) fp32 additions at 2^-24 relative.  A pair's
 * result does not depend on the rest of the batch or on table offsets.
 * gap_open, gap_extend > 0 and offset finite, else GFX_ERR_ARGUMENT; table
 * components must be finite (not checked here).
 * Workspace: gfx_align_workspace_bytes(P, m) serves every pair whose t_len is
 * at most m among those with q_len > 128 (the others need none).
 * ------------------------------------------------------------------------ */
size_t gfx_align_workspace_bytes(int64_t num_pairs, int64_t max_t_len);
int gfx_align(const void *queries, int64_t q_rows, const void *targets,
              int64_t t_rows, const int64_t *pairs, int64_t num_pairs,
              float offset, float gap_open, float gap_extend, float *out_score,
              int32_t *out_coords, void *workspace, size_t workspace_bytes,
              void *stream);

/* Traceback: gfx_align plus the aligned path of each pair.  Arguments,
 * argument errors and out_score / out_coords are those of gfx_align (the
 * messages name gfx_align_trace).
 * Ops, one byte per step in forward order (query_begin -> query_end):
 *   0 = M  query row i aligned with target row j (a diagonal step)
 *   1 = I  a query row against a gap (an F step, gap in the target)
 *   2 = D  a target row against a gap (an E step, gap in the query)
 * The path is the one the tie rules above define: from the end cell back,
 * H takes the first of diagonal, E, F that attains it, E and F prefer
 * opening to extending, and a diagonal step from H = 0 is the start.  It
 * starts and ends with M; #M + #I = query_end - query_begin and #M + #D =
 * target_end - target_begin, so it has at most (q_len + t_len - 1) ops.  A
 * pair with score 0 (or NaN) has an empty path.  Rescoring the path in fp32
 * reproduces the score bit for bit: v = 0 + s at the first M, then each M
 * adds its s, a gap opening (after M or after the other gap kind) subtracts
 * gap_open and an extension subtracts gap_extend.
 * out_ops uint8: pair p's path goes to out_ops[op_offsets[p] ...], a slot
 * the caller sizes to at least q_len + t_len - 1 bytes; op_offsets int64
 * [P]; out_len int32 [P] its length, or -1 if the walk did not end at the
 * reported start (a library bug; the path is then not written).
 * Workspace: gfx_align_trace_workspace_bytes(P, code_bytes), where
 * code_bytes >= sum over the pairs of q_len * ceil(t_len / 32) * 16 (4 bits
 * per cell of the DP's pointer record).  The per-CTA rows take every target
 * length, so no other property of the pairs enters the size.  Pointer
 * blocks are laid out in pair order; a pair whose block does not fit in the
 * workspace gets score NaN, like a pair outside the limits.
 * ------------------------------------------------------------------------ */
size_t gfx_align_trace_workspace_bytes(int64_t num_pairs, int64_t code_bytes);
int gfx_align_trace(const void *queries, int64_t q_rows, const void *targets,
                    int64_t t_rows, const int64_t *pairs, int64_t num_pairs,
                    float offset, float gap_open, float gap_extend,
                    float *out_score, int32_t *out_coords, uint8_t *out_ops,
                    const int64_t *op_offsets, int32_t *out_len,
                    void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * Instrumentation (used by bench.py; no effect on results).
 * Every kernel launch made by this library is counted per stage.  When a
 * stage's bit is set in the profile mask, each call of that stage is
 * bracketed by CUDA events on the launching stream; gfx_profile_read
 * synchronises those events and returns the summed device time.
 * ------------------------------------------------------------------------ */
enum {
  GFX_STAGE_PACK = 0,
  GFX_STAGE_CSR = 1,
  GFX_STAGE_CORE_ROWS = 2,
  GFX_STAGE_INPUT = 3,
  GFX_STAGE_AGGREGATE = 4,
  GFX_STAGE_MLP = 5,
  GFX_STAGE_HEAD = 6,
  GFX_STAGE_FUSED_LAYER = 7,
  GFX_STAGE_TOPK = 8,
  GFX_STAGE_BUILD = 9,
  GFX_STAGE_ALIGN = 10,
  GFX_NUM_STAGES = 11
};
int gfx_profile_enable(uint32_t stage_mask);
int gfx_profile_read(int stage, double *total_ms, int64_t *timed_calls, int reset);
int gfx_launch_counts(int64_t *counts /* [GFX_NUM_STAGES] */, int reset);

#ifdef __cplusplus
}
#endif
#endif /* GFX_H_ */
