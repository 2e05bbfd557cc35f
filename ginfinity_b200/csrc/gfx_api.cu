// Error plumbing, model upload and the whole-chunk forward driver.
#include <atomic>
#include <cstring>
#include <mutex>
#include <vector>

#include "gfx_common.cuh"

namespace gfx {

static thread_local std::string g_last_error;

void set_error(const std::string &msg) { g_last_error = msg; }
int fail(int code, const std::string &msg) {
  g_last_error = msg;
  return code;
}

// ---- instrumentation ----------------------------------------------------------
struct TimedCall { cudaEvent_t start, stop; int stage; };
static std::mutex g_prof_mutex;
static std::atomic<uint32_t> g_prof_mask{0};
static std::atomic<int64_t> g_launches[GFX_NUM_STAGES];
static std::vector<TimedCall> g_timed;          // recorded, not yet read
static std::vector<TimedCall> g_free;           // event pairs for reuse

StageScope::StageScope(int stage, cudaStream_t st, int launches) : st_(st), stop_(nullptr) {
  g_launches[stage].fetch_add(launches, std::memory_order_relaxed);
  if (!(g_prof_mask.load(std::memory_order_relaxed) & (1u << stage))) return;
  std::lock_guard<std::mutex> lock(g_prof_mutex);
  TimedCall c;
  if (!g_free.empty()) {
    c = g_free.back();
    g_free.pop_back();
  } else if (cudaEventCreate(&c.start) != cudaSuccess || cudaEventCreate(&c.stop) != cudaSuccess) {
    return;
  }
  c.stage = stage;
  cudaEventRecord(c.start, st);
  stop_ = c.stop;
  g_timed.push_back(c);
}

StageScope::~StageScope() {
  if (stop_) cudaEventRecord(stop_, st_);
}

// Round-trip through fp16 (round-to-nearest-even), on the host.
static inline float to_half_value(float v) { return __half2float(__float2half_rn(v)); }

// Append `count` floats to the arena image, 256-byte aligned; returns offset.
struct ArenaBuilder {
  std::vector<unsigned char> bytes;
  size_t reserve(size_t nbytes) {
    size_t off = (bytes.size() + 1023) & ~size_t(1023);
    bytes.resize(off + nbytes);
    return off;
  }
  size_t put(const std::vector<float> &v) {
    size_t off = reserve(v.size() * sizeof(float));
    std::memcpy(bytes.data() + off, v.data(), v.size() * sizeof(float));
    return off;
  }
  size_t put(const std::vector<__half> &v) {
    size_t off = reserve(v.size() * sizeof(__half));
    std::memcpy(bytes.data() + off, v.data(), v.size() * sizeof(__half));
    return off;
  }
};

// [rows][cols] -> [cols][rows]
static std::vector<float> transpose(const float *w, int rows, int cols, bool quantise) {
  std::vector<float> t(size_t(rows) * cols);
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < cols; ++c) {
      float v = w[size_t(r) * cols + c];
      t[size_t(c) * rows + r] = quantise ? to_half_value(v) : v;
    }
  return t;
}

static std::vector<float> copy(const float *w, size_t n, bool quantise) {
  std::vector<float> t(n);
  for (size_t i = 0; i < n; ++i) t[i] = quantise ? to_half_value(w[i]) : w[i];
  return t;
}

// K-major operand image for tcgen05.mma: W is [rows][k] row-major.  The image
// is k/64 consecutive tiles; tile kb holds columns [64kb, 64kb+64) as `rows`
// rows of 128 bytes whose eight 16-byte chunks are XOR-swizzled with (row&7)
// (the SWIZZLE_128B canonical layout; 8-row groups are 1024 bytes apart).
// `lo` selects the second part of the fp16 split w = hi + lo (hi = fp16(w), lo = fp16(w - hi)).
static void append_umma_image(std::vector<__half> &img, const float *w, int rows, int k, bool lo = false) {
  size_t base = img.size();
  img.resize(base + size_t(rows) * k);
  for (int kb = 0; kb < k / 64; ++kb)
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < 8; ++c)
        for (int j = 0; j < 8; ++j) {
          size_t dst = base + size_t(kb) * rows * 64 + size_t(r) * 64 + size_t((c ^ (r & 7)) * 8 + j);
          const float v = w[size_t(r) * k + kb * 64 + c * 8 + j];
          const __half hi = __float2half_rn(v);
          img[dst] = lo ? __float2half_rn(v - __half2float(hi)) : hi;
        }
}

}  // namespace gfx

using namespace gfx;

extern "C" int gfx_abi_version(void) { return GFX_ABI_VERSION; }
extern "C" const char *gfx_last_error(void) { return gfx::g_last_error.c_str(); }

extern "C" int gfx_profile_enable(uint32_t mask) {
  gfx::g_prof_mask.store(mask);
  return GFX_OK;
}

extern "C" int gfx_profile_read(int stage, double *total_ms, int64_t *timed_calls, int reset) {
  if (stage < 0 || stage >= GFX_NUM_STAGES) return fail(GFX_ERR_ARGUMENT, "gfx_profile_read: bad stage");
  std::lock_guard<std::mutex> lock(gfx::g_prof_mutex);
  double total = 0;
  int64_t calls = 0;
  std::vector<gfx::TimedCall> keep;
  for (auto &c : gfx::g_timed) {
    if (c.stage != stage) {
      keep.push_back(c);
      continue;
    }
    float ms = 0;
    GFX_CUDA(cudaEventSynchronize(c.stop));
    GFX_CUDA(cudaEventElapsedTime(&ms, c.start, c.stop));
    total += ms;
    ++calls;
    if (reset) gfx::g_free.push_back(c); else keep.push_back(c);
  }
  gfx::g_timed.swap(keep);
  if (total_ms) *total_ms = total;
  if (timed_calls) *timed_calls = calls;
  return GFX_OK;
}

extern "C" int gfx_launch_counts(int64_t *counts, int reset) {
  for (int s = 0; s < GFX_NUM_STAGES; ++s) {
    if (counts) counts[s] = gfx::g_launches[s].load();
    if (reset) gfx::g_launches[s].store(0);
  }
  return GFX_OK;
}

extern "C" int gfx_model_create(const gfx_folded_weights *w, gfx_model **out) {
  if (!w || !out) return fail(GFX_ERR_ARGUMENT, "gfx_model_create: null argument");
  if (w->hidden != kHidden || w->out_dim != kHidden || w->feature_dim != kFeat ||
      w->layers < 1 || w->layers > kMaxLayers || w->edge_dim < 1 || w->edge_dim > kMaxEdgeDim)
    return fail(GFX_ERR_UNSUPPORTED,
                "gfx_model_create: kernels are specialised for hidden=out_dim=128, "
                "feature_dim=7, layers<=8, edge_dim<=16");
  const int H = w->hidden, L = w->layers, M = 2 * H, F = w->feature_dim, ED = w->edge_dim;
  ArenaBuilder ab;
  size_t o_w_in[2], o_table[2], o_w1t[2], o_w2t[2], o_wat[2], o_wbt[2];
  for (int q = 0; q < 2; ++q) {
    o_w_in[q] = ab.put(copy(w->w_in_host, size_t(H) * F, q));
    o_table[q] = ab.put(copy(w->table_host, size_t(L) * ED * H, q));
    std::vector<float> t1, t2;
    for (int l = 0; l < L; ++l) {
      auto a = transpose(w->w1_host + size_t(l) * M * H, M, H, q);  // [H][2H]
      auto b = transpose(w->w2_host + size_t(l) * H * M, H, M, q);  // [2H][H]
      t1.insert(t1.end(), a.begin(), a.end());
      t2.insert(t2.end(), b.begin(), b.end());
    }
    o_w1t[q] = ab.put(t1);
    o_w2t[q] = ab.put(t2);
    o_wat[q] = ab.put(transpose(w->wa_host, H, H, q));
    o_wbt[q] = ab.put(transpose(w->wb_host, H, H, q));
  }
  size_t o_b_in = ab.put(copy(w->b_in_host, H, false));
  size_t o_b1 = ab.put(copy(w->b1_host, size_t(L) * M, false));
  size_t o_b2 = ab.put(copy(w->b2_host, size_t(L) * H, false));
  size_t o_g = ab.put(copy(w->ln_g_host, size_t(L) * H, false));
  size_t o_b = ab.put(copy(w->ln_b_host, size_t(L) * H, false));
  size_t o_ba = ab.put(copy(w->ba_host, H, false));
  size_t o_bb = ab.put(copy(w->bb_host, H, false));
  std::vector<__half> i1, i2, ia, ib;
  for (int l = 0; l < L; ++l) {
    append_umma_image(i1, w->w1_host + size_t(l) * M * H, M, H);
    append_umma_image(i2, w->w2_host + size_t(l) * H * M, H, M);
  }
  append_umma_image(ia, w->wa_host, H, H);
  append_umma_image(ib, w->wb_host, H, H);
  size_t o_i1 = ab.put(i1), o_i2 = ab.put(i2), o_ia = ab.put(ia), o_ib = ab.put(ib);
  std::vector<__half> l1, l2, la, lb;
  for (int l = 0; l < L; ++l) {
    append_umma_image(l1, w->w1_host + size_t(l) * M * H, M, H, true);
    append_umma_image(l2, w->w2_host + size_t(l) * H * M, H, M, true);
  }
  append_umma_image(la, w->wa_host, H, H, true);
  append_umma_image(lb, w->wb_host, H, H, true);
  size_t o_l1 = ab.put(l1), o_l2 = ab.put(l2), o_la = ab.put(la), o_lb = ab.put(lb);
  std::vector<__half> t16(size_t(L) * ED * H);
  for (size_t i = 0; i < t16.size(); ++i) t16[i] = __float2half_rn(w->table_host[i]);
  size_t o_t16 = ab.put(t16);

  gfx_model *m = new gfx_model();
  m->hidden = H; m->layers = L; m->out_dim = w->out_dim; m->feature_dim = F; m->edge_dim = ED;
  for (int l = 0; l < L; ++l) m->eps1[l] = w->eps1_host[l];
  m->host.b1.assign(w->b1_host, w->b1_host + size_t(L) * M);
  m->host.b2.assign(w->b2_host, w->b2_host + size_t(L) * H);
  m->host.ln_g.assign(w->ln_g_host, w->ln_g_host + size_t(L) * H);
  m->host.ln_b.assign(w->ln_b_host, w->ln_b_host + size_t(L) * H);
  m->host.ba.assign(w->ba_host, w->ba_host + H);
  m->host.bb.assign(w->bb_host, w->bb_host + H);
  cudaError_t err = cudaGetDevice(&m->device);
  if (err == cudaSuccess) err = cudaMalloc(&m->arena, ab.bytes.size());
  if (err == cudaSuccess)
    err = cudaMemcpy(m->arena, ab.bytes.data(), ab.bytes.size(), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    delete m;
    return fail(GFX_ERR_CUDA, std::string("gfx_model_create: ") + cudaGetErrorString(err));
  }
  auto f = [&](size_t off) { return reinterpret_cast<const float *>(static_cast<char *>(m->arena) + off); };
  auto h = [&](size_t off) { return reinterpret_cast<const __half *>(static_cast<char *>(m->arena) + off); };
  for (int q = 0; q < 2; ++q) {
    m->w_in[q] = f(o_w_in[q]); m->table[q] = f(o_table[q]);
    m->w1t[q] = f(o_w1t[q]); m->w2t[q] = f(o_w2t[q]);
    m->wat[q] = f(o_wat[q]); m->wbt[q] = f(o_wbt[q]);
  }
  m->b_in = f(o_b_in); m->b1 = f(o_b1); m->b2 = f(o_b2); m->ln_g = f(o_g); m->ln_b = f(o_b);
  m->ba = f(o_ba); m->bb = f(o_bb);
  m->w1_img = h(o_i1); m->w2_img = h(o_i2); m->wa_img = h(o_ia); m->wb_img = h(o_ib); m->table16 = h(o_t16);
  m->w1_lo_img = h(o_l1); m->w2_lo_img = h(o_l2); m->wa_lo_img = h(o_la); m->wb_lo_img = h(o_lb);
  *out = m;
  return GFX_OK;
}

extern "C" int gfx_model_destroy(gfx_model *m) {
  if (!m) return GFX_OK;
  cudaFree(m->arena);
  delete m;
  return GFX_OK;
}

// ---------------------------------------------------------------------------
// Whole forward over one chunk: input linear, `layers` x (aggregate, MLP) or
// fused layers, head + L2 normalise.  Workspace: 3 activation buffers.
// ---------------------------------------------------------------------------
static size_t act_bytes(int64_t n, int dtype) {
  size_t e = dtype == GFX_F16 ? 2 : 4;
  return (size_t(n) * kHidden * e + 1023) & ~size_t(1023);
}

extern "C" size_t gfx_encode_workspace_bytes(int64_t num_nodes, int dtype) {
  return 3 * act_bytes(num_nodes, dtype);
}

static int encode_chunk(const gfx_model *model, const float *x, const int32_t *row_ptr,
                        const int32_t *col_src, const uint8_t *col_type, const uint32_t *desc_in,
                        const int32_t *needs_csr, const int32_t *out_row, int64_t n, void *out, int dtype, int out_dtype, int impl,
                        int fused, void *ws, size_t ws_bytes, void *stream);

extern "C" int gfx_encode(const gfx_model *model, const float *x, const int32_t *row_ptr,
                          const int32_t *col_src, const uint8_t *col_type,
                          const int32_t *out_row, int64_t n, void *out, int dtype,
                          int out_dtype, int impl, int fused, void *ws, size_t ws_bytes,
                          void *stream) {
  return encode_chunk(model, x, row_ptr, col_src, col_type, nullptr, nullptr, out_row, n, out, dtype,
                      out_dtype, impl, fused, ws, ws_bytes, stream);
}

extern "C" int gfx_encode_described(const gfx_model *model, const float *x, const uint32_t *desc,
                                    const int32_t *row_ptr, const int32_t *col_src,
                                    const uint8_t *col_type, int64_t n, void *out, int out_dtype,
                                    void *ws, size_t ws_bytes, void *stream) {
  if (!desc && n > 0) return fail(GFX_ERR_ARGUMENT, "gfx_encode_described: null row descriptors");
  return encode_chunk(model, x, row_ptr, col_src, col_type, desc, nullptr, nullptr, n, out, GFX_F16,
                      out_dtype, GFX_IMPL_AUTO, 3, ws, ws_bytes, stream);
}

extern "C" int gfx_encode_described_f32(const gfx_model *model, const float *x, const uint32_t *desc,
                                        const int32_t *needs_csr, const int32_t *row_ptr,
                                        const int32_t *col_src, const uint8_t *col_type, int64_t n,
                                        void *out, int out_dtype, void *ws, size_t ws_bytes,
                                        void *stream) {
  if ((!desc || !needs_csr) && n > 0)
    return fail(GFX_ERR_ARGUMENT, "gfx_encode_described_f32: null row descriptors or flag");
  return encode_chunk(model, x, row_ptr, col_src, col_type, desc, needs_csr, nullptr, n, out, GFX_F32,
                      out_dtype, GFX_IMPL_AUTO, 0, ws, ws_bytes, stream);
}

static int encode_chunk(const gfx_model *model, const float *x, const int32_t *row_ptr,
                        const int32_t *col_src, const uint8_t *col_type, const uint32_t *desc_in,
                        const int32_t *needs_csr, const int32_t *out_row, int64_t n, void *out, int dtype, int out_dtype, int impl,
                        int fused, void *ws, size_t ws_bytes, void *stream) {
  if (!model) return fail(GFX_ERR_ARGUMENT, "gfx_encode: null model");
  if (n == 0) return GFX_OK;
  if (ws_bytes < gfx_encode_workspace_bytes(n, dtype))
    return fail(GFX_ERR_WORKSPACE, "gfx_encode: workspace too small");
  if (fused < 0 || fused > 3) return fail(GFX_ERR_ARGUMENT, "gfx_encode: fused must be 0, 2 or 3");
  if (fused && dtype != GFX_F16)
    return fail(GFX_ERR_UNSUPPORTED, "gfx_encode: fused layers exist for GFX_F16 only");
  if (fused == 1) fused = 2;   // the one-CTA-per-SM form was removed; 1 is kept as an alias
  // the banded kernel covers >= 6 edge types and <= 2^25 nodes, the CTA-pair kernel <= 10 edge
  // types and <= 2^27 nodes; outside that: K1 + K2
  if (desc_in != nullptr && (model->edge_dim < 6 || n > (int64_t(1) << 25)))
    return fail(GFX_ERR_UNSUPPORTED, "gfx_encode_described: needs >= 6 edge types and <= 2^25 nodes");
  if (fused == 3 && (model->edge_dim < 6 || n > (int64_t(1) << 25))) fused = 2;
  if (fused == 2 && (model->edge_dim > 10 || n > (int64_t(1) << 27))) fused = 0;
  char *base = static_cast<char *>(ws);
  void *h = base, *z = base + act_bytes(n, dtype), *h2 = base + 2 * act_bytes(n, dtype);
  int rc = gfx_input_linear(model, x, n, h, dtype, stream);
  if (rc) return rc;
  const uint32_t *desc = desc_in;
  if (fused == 3 && desc == nullptr) {
    uint32_t *made = static_cast<uint32_t *>(z);     // fused layers leave the z buffer free
    rc = gfx_row_describe(row_ptr, col_src, col_type, n, made, stream);
    if (rc) return rc;
    desc = made;
  }
  for (int l = 0; l < model->layers; ++l) {
    if (fused == 3) {   // CTA pairs, banded producers (gfx_fused8.cu)
      rc = gfx_layer_fused_banded(model, l, h, row_ptr, col_src, col_type, desc, n, h2, stream);
      if (rc) return rc;
    } else if (fused) {   // CTA pairs, producers walk the CSR arrays (gfx_fused6.cu)
      rc = gfx_layer_fused_pair(model, l, h, row_ptr, col_src, col_type, n, h2, stream);
      if (rc) return rc;
    } else {
      rc = (desc_in != nullptr && dtype == GFX_F32)
               ? gfx_aggregate_banded(model, l, h, desc_in, needs_csr, row_ptr, col_src, col_type, n, z,
                                      dtype, stream)
               : gfx_aggregate(model, l, h, row_ptr, col_src, col_type, n, z, dtype, stream);
      if (rc) return rc;
      rc = gfx_mlp_ln_residual(model, l, z, h, n, h2, dtype, impl, stream);
      if (rc) return rc;
    }
    void *t = h; h = h2; h2 = t;
  }
  return gfx_head_l2norm(model, h, out_row, n, out, dtype, out_dtype, impl, stream);
}
