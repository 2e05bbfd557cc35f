// CUDA-core kernels: input projection, K1 neighbour aggregation (the HBM-bound
// kernel of the path) and an fp32-accumulate MLP / head used for the
// full-precision model and as the on-device cross-check of the tcgen05 path.
#include "gfx_common.cuh"
#include "gfx_umma.cuh"

namespace gfx {

// ---- 8-channel row slices ---------------------------------------------------
// A node row is 128 channels.  A half-warp (16 lanes) owns one row; lane l
// owns channels [8l, 8l+8): 16 bytes of fp16 (one 128-bit access) or 32 bytes
// of fp32 (two 128-bit accesses), so a row is read with full 128-byte lines.
struct Row8 {
  float v[8];
};

__device__ __forceinline__ Row8 load8(const __half *p) {
  uint4 raw = *reinterpret_cast<const uint4 *>(p);
  const __half2 *h = reinterpret_cast<const __half2 *>(&raw);
  Row8 r;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __half22float2(h[i]);
    r.v[2 * i] = f.x;
    r.v[2 * i + 1] = f.y;
  }
  return r;
}
__device__ __forceinline__ Row8 load8(const float *p) {
  float4 a = reinterpret_cast<const float4 *>(p)[0];
  float4 b = reinterpret_cast<const float4 *>(p)[1];
  return Row8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
__device__ __forceinline__ void store8(__half *p, const Row8 &r) {
  uint4 raw;
  __half2 *h = reinterpret_cast<__half2 *>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(r.v[2 * i], r.v[2 * i + 1]);
  *reinterpret_cast<uint4 *>(p) = raw;
}
__device__ __forceinline__ void store8(float *p, const Row8 &r) {
  reinterpret_cast<float4 *>(p)[0] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  reinterpret_cast<float4 *>(p)[1] = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
}

// ---------------------------------------------------------------------------
// input projection  h = x W_in^T + b_in     (28 B in, 256/512 B out per node)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
input_linear_kernel(const float *__restrict__ x, const float *__restrict__ w_in,
                    const float *__restrict__ b_in, int64_t n, T *__restrict__ h) {
  const int sub = threadIdx.x & 15;                 // lane within the half-warp
  float w[8][kFeat], b[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    b[c] = b_in[sub * 8 + c];
#pragma unroll
    for (int f = 0; f < kFeat; ++f) w[c][f] = w_in[(sub * 8 + c) * kFeat + f];
  }
  const int64_t rows_per_pass = int64_t(gridDim.x) * (blockDim.x >> 4);
  for (int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4); i < n;
       i += rows_per_pass) {
    float xf[kFeat];
#pragma unroll
    for (int f = 0; f < kFeat; ++f) xf[f] = x[i * kFeat + f];
    Row8 r;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float acc = b[c];
#pragma unroll
      for (int f = 0; f < kFeat; ++f) acc = fmaf(xf[f], w[c][f], acc);
      r.v[c] = acc;
    }
    store8(h + i * kHidden + sub * 8, r);
  }
}

// Four consecutive nodes per half-warp and iteration: their 28 features are
// seven 128-bit loads issued up front (x must be 16-byte aligned), so the
// kernel runs at the speed of its 256 B/node of stores instead of waiting on
// seven dependent scalar loads per node.
template <typename T>
__global__ void __launch_bounds__(256)
input_linear4_kernel(const float *__restrict__ x, const float *__restrict__ w_in,
                     const float *__restrict__ b_in, int64_t n, T *__restrict__ h) {
  const int sub = threadIdx.x & 15;
  float w[8][kFeat], b[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    b[c] = b_in[sub * 8 + c];
#pragma unroll
    for (int f = 0; f < kFeat; ++f) w[c][f] = w_in[(sub * 8 + c) * kFeat + f];
  }
  const int64_t groups = (n + 3) / 4;
  const int64_t per_pass = int64_t(gridDim.x) * (blockDim.x >> 4);
  for (int64_t g = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4); g < groups;
       g += per_pass) {
    const int64_t i0 = g * 4;
    float xf[4 * kFeat];
    if (i0 + 4 <= n) {
      const float4 *xv = reinterpret_cast<const float4 *>(x + i0 * kFeat);
#pragma unroll
      for (int q = 0; q < kFeat; ++q) {
        const float4 v = xv[q];
        xf[4 * q] = v.x; xf[4 * q + 1] = v.y; xf[4 * q + 2] = v.z; xf[4 * q + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 4 * kFeat; ++q) xf[q] = i0 * kFeat + q < n * kFeat ? x[i0 * kFeat + q] : 0.f;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      Row8 o;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float acc = b[c];
#pragma unroll
        for (int f = 0; f < kFeat; ++f) acc = fmaf(xf[r * kFeat + f], w[c][f], acc);
        o.v[c] = acc;
      }
      if (i0 + r < n) store8(h + (i0 + r) * kHidden + sub * 8, o);
    }
  }
}

// ---------------------------------------------------------------------------
// K1  z_i = eps1 * h_i + sum_{e in row i} relu(h[col_src[e]] + table[col_type[e]])
// One half-warp per destination node, edges of a row taken four at a time so
// that four independent 128-bit row loads are in flight per lane.  Sums are
// fp32 in CSR order (= reference edge order), so the result is deterministic.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
aggregate_kernel(const T *__restrict__ h, const int32_t *__restrict__ row_ptr,
                 const int32_t *__restrict__ col_src, const uint8_t *__restrict__ col_type,
                 const float *__restrict__ table, int edge_dim, float eps1, int64_t n,
                 T *__restrict__ z) {
  __shared__ __align__(16) float tab[kMaxEdgeDim * kHidden];
  for (int i = threadIdx.x; i < edge_dim * kHidden; i += blockDim.x) tab[i] = table[i];
  __syncthreads();
  const int sub = threadIdx.x & 15;
  const int64_t rows_per_pass = int64_t(gridDim.x) * (blockDim.x >> 4);
  for (int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4); i < n;
       i += rows_per_pass) {
    const int beg = row_ptr[i], end = row_ptr[i + 1];
    Row8 self = load8(h + i * kHidden + sub * 8);
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    int e = beg;
    for (; e + 4 <= end; e += 4) {
      int s[4], t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s[u] = col_src[e + u];
        t[u] = col_type[e + u];
      }
      Row8 nb[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) nb[u] = load8(h + int64_t(s[u]) * kHidden + sub * 8);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float *tp = tab + t[u] * kHidden + sub * 8;
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] += fmaxf(nb[u].v[c] + tp[c], 0.f);
      }
    }
    for (; e < end; ++e) {
      const int s = col_src[e], t = col_type[e];
      Row8 nb = load8(h + int64_t(s) * kHidden + sub * 8);
      const float *tp = tab + t * kHidden + sub * 8;
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[c] += fmaxf(nb.v[c] + tp[c], 0.f);
    }
    Row8 out;
#pragma unroll
    for (int c = 0; c < 8; ++c) out.v[c] = fmaf(eps1, self.v[c], acc[c]);
    store8(z + i * kHidden + sub * 8, out);
  }
}

// ---------------------------------------------------------------------------
// K1, fp16 storage: the same half-warp-per-node scheme with packed math.  The
// message relu(h_src + table[type]) is one HFMA2.RELU per channel pair
// (rounded to fp16, which is what the reference's own fp16 path does,
// _model.py:43); the sum stays fp32 via the mixed-precision add
// (add.rn.f32.f16 -> FHADD), in CSR order.  1.5 instructions per channel and
// edge instead of 4, and the fp16 table row is one conflict-free 128-bit
// shared-memory load per edge.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hfma2_relu_add(uint32_t x, uint32_t t) {
  uint32_t r;
  asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0x3c003c00u), "r"(t));
  return r;
}
__device__ __forceinline__ void add_pair(float &a0, float &a1, uint32_t m) {
  asm("{\n.reg .b16 lo, hi;\nmov.b32 {lo, hi}, %2;\nadd.rn.f32.f16 %0, lo, %0;\n"
      "add.rn.f32.f16 %1, hi, %1;\n}"
      : "+f"(a0), "+f"(a1)
      : "r"(m));
}
__device__ __forceinline__ void add_message(float *acc, const uint4 &nb, const uint4 &tb) {
  add_pair(acc[0], acc[1], hfma2_relu_add(nb.x, tb.x));
  add_pair(acc[2], acc[3], hfma2_relu_add(nb.y, tb.y));
  add_pair(acc[4], acc[5], hfma2_relu_add(nb.z, tb.z));
  add_pair(acc[6], acc[7], hfma2_relu_add(nb.w, tb.w));
}

// The per-node chain row_ptr -> col_src/col_type -> neighbour rows is three
// dependent memory latencies; run naively a half-warp spends two thirds of its
// time with ~100 bytes in flight.  The loop below is software-pipelined two
// nodes deep: while node i's rows are in flight, node i+1's edge indices and
// node i+2's row_ptr entries are being fetched, so every resident half-warp
// always has its ~1.5 KB of row loads outstanding.  kWin edges per node are
// covered by the pipeline (the builder's graphs have in-degree <= 5); longer
// rows finish in a plain loop.
constexpr int kWin = 5;

__device__ __forceinline__ void load_window(const int32_t *__restrict__ col_src,
                                            const uint8_t *__restrict__ col_type, int beg, int end,
                                            int *s, int *t) {
#pragma unroll
  for (int u = 0; u < kWin; ++u) {
    const bool ok = beg + u < end;
    s[u] = ok ? col_src[beg + u] : 0;
    t[u] = ok ? int(col_type[beg + u]) : 0;
  }
}

__global__ void __launch_bounds__(256, 4)
aggregate_f16_kernel(const __half *__restrict__ h, const int32_t *__restrict__ row_ptr,
                     const int32_t *__restrict__ col_src, const uint8_t *__restrict__ col_type,
                     const __half *__restrict__ table16, int edge_dim, float eps1, int64_t n,
                     __half *__restrict__ z) {
  __shared__ __align__(16) __half tab[kMaxEdgeDim * kHidden];
  for (int i = threadIdx.x; i < edge_dim * kHidden / 8; i += blockDim.x)
    reinterpret_cast<uint4 *>(tab)[i] = reinterpret_cast<const uint4 *>(table16)[i];
  __syncthreads();
  const int sub = threadIdx.x & 15;
  const uint4 *hv = reinterpret_cast<const uint4 *>(h) + sub;      // row r -> hv[r * 16]
  const uint4 *tv = reinterpret_cast<const uint4 *>(tab) + sub;
  const int64_t stride = int64_t(gridDim.x) * (blockDim.x >> 4);
  // Nodes are visited from the END of the chunk towards its start: K2 (ascending)
  // wrote the last rows of h most recently, and the z rows written last here (the
  // start of the chunk) are the first ones K2 reads -- both while still in L2.
  // `i` counts visits; the node is n-1-i.
  int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4);
  if (i >= n) return;
  const int64_t last = n - 1;
  int beg = row_ptr[last - i], end = row_ptr[last - i + 1];
  int64_t i1 = i + stride;
  int beg1 = 0, end1 = 0;
  if (i1 < n) {
    beg1 = row_ptr[last - i1];
    end1 = row_ptr[last - i1 + 1];
  }
  int s[kWin], t[kWin];
  load_window(col_src, col_type, beg, end, s, t);
  while (true) {
    const int64_t i2 = i1 + stride;
    int beg2 = 0, end2 = 0;
    if (i2 < n) {                                   // stage 1: row_ptr two nodes ahead
      beg2 = row_ptr[last - i2];
      end2 = row_ptr[last - i2 + 1];
    }
    int s1[kWin], t1[kWin];
    load_window(col_src, col_type, beg1, end1, s1, t1);   // stage 2: indices one node ahead
    const uint4 self = hv[(last - i) * 16];         // stage 3: this node's rows
    const int deg = end - beg;
    uint4 nb[kWin];
#pragma unroll
    for (int u = 0; u < kWin; ++u) nb[u] = u < deg ? hv[int64_t(s[u]) * 16] : make_uint4(0, 0, 0, 0);
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
#pragma unroll
    for (int u = 0; u < kWin; ++u)
      if (u < deg) add_message(acc, nb[u], tv[t[u] * 16]);
    for (int e = beg + kWin; e < end; ++e)          // rows longer than the window
      add_message(acc, hv[int64_t(col_src[e]) * 16], tv[int(col_type[e]) * 16]);
    const __half2 *sh = reinterpret_cast<const __half2 *>(&self);
    uint4 out;
    uint32_t *o = reinterpret_cast<uint32_t *>(&out);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float2 f = __half22float2(sh[c]);
      const __half2 r = __floats2half2_rn(fmaf(eps1, f.x, acc[2 * c]), fmaf(eps1, f.y, acc[2 * c + 1]));
      o[c] = *reinterpret_cast<const uint32_t *>(&r);
    }
    reinterpret_cast<uint4 *>(z)[(last - i) * 16 + sub] = out;
    if (i1 >= n) break;
    i = i1; beg = beg1; end = end1;
    i1 = i2; beg1 = beg2; end1 = end2;
#pragma unroll
    for (int u = 0; u < kWin; ++u) {
      s[u] = s1[u];
      t[u] = t1[u];
    }
  }
}

// ---------------------------------------------------------------------------
// K1, fp16 storage, quarter-warp per node.  ncu of the half-warp kernel above
// (profiles/r01_f): 71 % of the issue slots busy at 39 % of DRAM throughput,
// 120 warp instructions per node -- it is bound by instruction issue, and half
// of what it issues is per-node bookkeeping (index loads with their address
// arithmetic, divergent `u < deg` regions) that costs the same for 16 lanes
// as for 8.  Here 8 lanes own a node (lane q: channels [8q, 8q+8) and
// [64+8q, 64+8q+8), i.e. two 128-bit accesses, each instruction covering a
// contiguous 128-byte line per node), so a warp retires 4 nodes per pass
// through the same bookkeeping:
//   * lane q fetches edge `beg + q` (source and type, packed into one
//     register) and the 8 lanes exchange them by shuffle: 2 loads + 5 SHFL
//     instead of 10 loads;
//   * a missing edge (u >= deg) points at the node itself with a table row of
//     -65504, so its message is relu(h - 65504) = +0 and nothing is
//     predicated or divergent; the extra row read is an L1 hit (the self row
//     is loaded anyway);
//   * the software pipeline is the same (row_ptr two nodes ahead, indices one
//     node ahead, rows now).
// Rows with more than 8 edges finish in a plain loop.  Sources must fit 27
// bits (the caller falls back to the half-warp kernel above 2^27 nodes).
// 4 resident blocks per SM (64 registers, no spills): 0.074 ms on a 603k-node
// chunk against 0.081 ms at 2 blocks (115 registers).
// ---------------------------------------------------------------------------
constexpr int kWinQ = 5;              // edges per node covered by the straight-line code
constexpr int kSrcBits = 27;
constexpr uint32_t kSrcMask = (1u << kSrcBits) - 1u;

__global__ void __launch_bounds__(256, 4)
aggregate_f16_q_kernel(const __half *__restrict__ h, const int32_t *__restrict__ row_ptr,
                       const int32_t *__restrict__ col_src, const uint8_t *__restrict__ col_type,
                       const __half *__restrict__ table16, int edge_dim, float eps1, int64_t n,
                       __half *__restrict__ z) {
  __shared__ __align__(16) __half tab[(kMaxEdgeDim + 1) * kHidden];
  for (int i = threadIdx.x; i < edge_dim * kHidden / 8; i += blockDim.x)
    reinterpret_cast<uint4 *>(tab)[i] = reinterpret_cast<const uint4 *>(table16)[i];
  for (int i = threadIdx.x; i < kHidden / 8; i += blockDim.x)       // the "no edge" row
    reinterpret_cast<uint4 *>(tab)[edge_dim * kHidden / 8 + i] =
        make_uint4(0xFBFFFBFFu, 0xFBFFFBFFu, 0xFBFFFBFFu, 0xFBFFFBFFu);
  __syncthreads();
  const int sub = threadIdx.x & 7;
  const int qbase = threadIdx.x & 24;                               // first lane of this quarter
  const uint4 *hv = reinterpret_cast<const uint4 *>(h) + sub;       // row r -> hv[r*16], hv[r*16+8]
  const uint4 *tv = reinterpret_cast<const uint4 *>(tab) + sub;
  const uint32_t none = uint32_t(edge_dim) << kSrcBits;
  const int64_t stride = int64_t(gridDim.x) * (blockDim.x >> 3);
  // descending node order, as in the half-warp kernel (L2 hand-over with K2)
  int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 3) + (threadIdx.x >> 3);
  const int64_t last = n - 1;
  // Out-of-range quarters keep running with an empty row (every shuffle below
  // is executed by the full warp) and skip only the store.
  auto rp = [&](int64_t v, int &b, int &e) {
    b = e = 0;
    if (v < n) {
      b = row_ptr[last - v];
      e = row_ptr[last - v + 1];
    }
  };
  auto fetch_edge = [&](int64_t v, int b, int e) -> uint32_t {       // this lane's edge of node v
    uint32_t pk = (uint32_t(v < n ? last - v : 0) & kSrcMask) | none;
    if (b + sub < e) pk = uint32_t(col_src[b + sub]) | (uint32_t(col_type[b + sub]) << kSrcBits);
    return pk;
  };
  int beg, end, beg1, end1;
  rp(i, beg, end);
  int64_t i1 = i + stride;
  rp(i1, beg1, end1);
  uint32_t pk = fetch_edge(i, beg, end);
  while (true) {                                                     // warp-uniform trip count
    const int64_t i2 = i1 + stride;
    int beg2, end2;
    rp(i2, beg2, end2);                                              // stage 1
    const uint32_t pk1 = fetch_edge(i1, beg1, end1);                 // stage 2
    const int64_t node = i < n ? last - i : 0;                       // stage 3
    const uint4 self0 = hv[node * 16], self1 = hv[node * 16 + 8];
    uint32_t e[kWinQ];
    uint4 nb0[kWinQ], nb1[kWinQ];
#pragma unroll
    for (int u = 0; u < kWinQ; ++u) {
      e[u] = __shfl_sync(0xffffffffu, pk, qbase + u);
      const uint4 *src = hv + int64_t(e[u] & kSrcMask) * 16;
      nb0[u] = src[0];
      nb1[u] = src[8];
    }
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = 0.f;
#pragma unroll
    for (int u = 0; u < kWinQ; ++u) {
      const uint4 *t = tv + (e[u] >> kSrcBits) * 16;
      add_message(acc, nb0[u], t[0]);
      add_message(acc + 8, nb1[u], t[8]);
    }
    const int deg = end - beg;
    if (deg > kWinQ) {                                               // rare: longer rows
      for (int u = kWinQ; u < deg; ++u) {
        const int s = col_src[beg + u], ty = col_type[beg + u];
        const uint4 *src = hv + int64_t(s) * 16;
        const uint4 *t = tv + ty * 16;
        add_message(acc, src[0], t[0]);
        add_message(acc + 8, src[8], t[8]);
      }
    }
    if (i < n) {
      uint4 o0, o1;
      uint32_t *p0 = reinterpret_cast<uint32_t *>(&o0), *p1 = reinterpret_cast<uint32_t *>(&o1);
      const __half2 *s0 = reinterpret_cast<const __half2 *>(&self0);
      const __half2 *s1 = reinterpret_cast<const __half2 *>(&self1);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float2 f0 = __half22float2(s0[c]), f1 = __half22float2(s1[c]);
        const __half2 r0 = __floats2half2_rn(fmaf(eps1, f0.x, acc[2 * c]), fmaf(eps1, f0.y, acc[2 * c + 1]));
        const __half2 r1 =
            __floats2half2_rn(fmaf(eps1, f1.x, acc[8 + 2 * c]), fmaf(eps1, f1.y, acc[8 + 2 * c + 1]));
        p0[c] = *reinterpret_cast<const uint32_t *>(&r0);
        p1[c] = *reinterpret_cast<const uint32_t *>(&r1);
      }
      uint4 *zr = reinterpret_cast<uint4 *>(z) + node * 16 + sub;
      zr[0] = o0;
      zr[8] = o1;
    }
    // the first node of the warp is the lowest visit index: all four are done when it is
    if (__shfl_sync(0xffffffffu, int(i1 >= n), 0)) break;
    i = i1; beg = beg1; end = end1; pk = pk1;
    i1 = i2; beg1 = beg2; end1 = end2;
  }
}

// ---------------------------------------------------------------------------
// K1, fp32 storage (full_precision): the quarter-warp scheme above with a HALF warp per node (a
// 512-byte row is 16 lanes x two 128-bit loads), edges fetched by one lane each and exchanged by
// shuffle, a missing edge pointing at the node itself with a -FLT_MAX table row (message +0),
// software-pipelined two nodes deep.  Same operations in the same order as aggregate_kernel<float>
// (fp32 message, fp32 sum in CSR order, one fma for the self term): the same bits.
// ---------------------------------------------------------------------------
constexpr int kWinH = 5;

__global__ void __launch_bounds__(256, 2)
aggregate_f32_h_kernel(const float *__restrict__ h, const int32_t *__restrict__ row_ptr,
                       const int32_t *__restrict__ col_src, const uint8_t *__restrict__ col_type,
                       const float *__restrict__ table, int edge_dim, float eps1, int64_t n,
                       float *__restrict__ z, const int32_t *__restrict__ gate) {
  if (gate != nullptr && *gate == 0) return;     // gfx_aggregate_banded: the banded kernel did the chunk
  __shared__ __align__(16) float tab[(kMaxEdgeDim + 1) * kHidden];
  for (int i = threadIdx.x; i < edge_dim * kHidden; i += blockDim.x) tab[i] = table[i];
  for (int i = threadIdx.x; i < kHidden; i += blockDim.x) tab[edge_dim * kHidden + i] = -3.0e38f;
  __syncthreads();
  const int sub = threadIdx.x & 15;
  const int hbase = threadIdx.x & 16;                               // first lane of this half warp
  const float4 *hv = reinterpret_cast<const float4 *>(h) + sub;     // row r -> hv[r*32], hv[r*32+16]
  const float4 *tv = reinterpret_cast<const float4 *>(tab) + sub;
  const uint32_t none = uint32_t(edge_dim) << kSrcBits;
  const int64_t stride = int64_t(gridDim.x) * (blockDim.x >> 4);
  int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4);
  const int64_t last = n - 1;                                        // descending node order (L2 hand-over)
  auto rp = [&](int64_t v, int &b, int &e) {
    b = e = 0;
    if (v < n) {
      b = row_ptr[last - v];
      e = row_ptr[last - v + 1];
    }
  };
  auto fetch_edge = [&](int64_t v, int b, int e) -> uint32_t {       // this lane's edge of node v
    uint32_t pk = (uint32_t(v < n ? last - v : 0) & kSrcMask) | none;
    if (b + sub < e) pk = uint32_t(col_src[b + sub]) | (uint32_t(col_type[b + sub]) << kSrcBits);
    return pk;
  };
  int beg, end, beg1, end1;
  rp(i, beg, end);
  int64_t i1 = i + stride;
  rp(i1, beg1, end1);
  uint32_t pk = fetch_edge(i, beg, end);
  while (true) {                                                     // warp-uniform trip count
    const int64_t i2 = i1 + stride;
    int beg2, end2;
    rp(i2, beg2, end2);
    const uint32_t pk1 = fetch_edge(i1, beg1, end1);
    const int64_t node = i < n ? last - i : 0;
    const float4 self0 = hv[node * 32], self1 = hv[node * 32 + 16];
    uint32_t e[kWinH];
    float4 nb0[kWinH], nb1[kWinH];
#pragma unroll
    for (int u = 0; u < kWinH; ++u) {
      e[u] = __shfl_sync(0xffffffffu, pk, hbase + u);
      const float4 *src = hv + int64_t(e[u] & kSrcMask) * 32;
      nb0[u] = src[0];
      nb1[u] = src[16];
    }
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    auto add = [&](const float4 &a, const float4 &b, const float4 &t0, const float4 &t1) {
      acc[0] += fmaxf(a.x + t0.x, 0.f); acc[1] += fmaxf(a.y + t0.y, 0.f);
      acc[2] += fmaxf(a.z + t0.z, 0.f); acc[3] += fmaxf(a.w + t0.w, 0.f);
      acc[4] += fmaxf(b.x + t1.x, 0.f); acc[5] += fmaxf(b.y + t1.y, 0.f);
      acc[6] += fmaxf(b.z + t1.z, 0.f); acc[7] += fmaxf(b.w + t1.w, 0.f);
    };
#pragma unroll
    for (int u = 0; u < kWinH; ++u) {
      const float4 *t = tv + (e[u] >> kSrcBits) * 32;
      add(nb0[u], nb1[u], t[0], t[16]);
    }
    const int deg = end - beg;
    if (deg > kWinH) {                                               // rare: longer rows
      for (int u = kWinH; u < deg; ++u) {
        const int s = col_src[beg + u], ty = col_type[beg + u];
        const float4 *src = hv + int64_t(s) * 32;
        const float4 *t = tv + ty * 32;
        add(src[0], src[16], t[0], t[16]);
      }
    }
    if (i < n) {
      float4 *zr = reinterpret_cast<float4 *>(z) + node * 32 + sub;
      zr[0] = make_float4(fmaf(eps1, self0.x, acc[0]), fmaf(eps1, self0.y, acc[1]),
                          fmaf(eps1, self0.z, acc[2]), fmaf(eps1, self0.w, acc[3]));
      zr[16] = make_float4(fmaf(eps1, self1.x, acc[4]), fmaf(eps1, self1.y, acc[5]),
                           fmaf(eps1, self1.z, acc[6]), fmaf(eps1, self1.w, acc[7]));
    }
    if (__shfl_sync(0xffffffffu, int(i1 >= n), 0)) break;
    i = i1; beg = beg1; end = end1; pk = pk1;
    i1 = i2; beg1 = beg2; end1 = end2;
  }
}

// ---------------------------------------------------------------------------
// K1, fp32 storage, from ROW DESCRIPTORS (gfx_edge_describe): when every row of the chunk is one
// of the reference builder's banded rows -- (i-1) (i+1) [(partner)] (i-2) (i+2), some missing at
// molecule ends -- a block walks tiles of 64 consecutive rows.  A tile and its two halo rows on
// either side (68 x 512 bytes, contiguous in h) arrive in shared memory by ONE bulk copy on the
// TMA engine, three tiles deep (two in flight while one is computed: ~70 KB per block on the way
// without holding registers); a warp owns 8 rows of the tile, one float4 per lane, slides a
// five-row register window over them (one LDS.128 per row) and fetches only the pairing partners
// from global memory, all eight up front (prefetched into L2 a tile ahead).  Each h row crosses
// the LSU once instead of once per edge (the CSR kernel above is bound by the L1 / LSU pipe:
// 3.5 KB per node through it, 84 % busy in ncu).  Same operations in the same order as the CSR
// kernels (fp32 message, fp32 sum in CSR order with a missing edge adding nothing, one fma for
// the self term): the same bits.  Runs only when *gate == 0 (no GENERIC row in the chunk);
// otherwise the CSR kernel does the chunk.
// ---------------------------------------------------------------------------
constexpr int kBandTile = 64, kBandStages = 3;
constexpr int kBandStageBytes = (kBandTile + 4) * kHidden * 4;
constexpr int kBandSmemBytes = kBandStages * kBandStageBytes + 64;

__device__ __forceinline__ void band_add(float4 &acc, const float4 &a, const float4 &t) {
  acc.x += fmaxf(a.x + t.x, 0.f);
  acc.y += fmaxf(a.y + t.y, 0.f);
  acc.z += fmaxf(a.z + t.z, 0.f);
  acc.w += fmaxf(a.w + t.w, 0.f);
}

__global__ void __launch_bounds__(256, 2)
aggregate_f32_band_kernel(const float *__restrict__ h, const uint32_t *__restrict__ desc,
                          const int32_t *__restrict__ gate, const float *__restrict__ table,
                          float eps1, int n, float *__restrict__ z) {
  using namespace rowdesc;
  using namespace ptx;
  extern __shared__ __align__(128) unsigned char band_smem[];
  if (*gate != 0) return;
  uint64_t *full = reinterpret_cast<uint64_t *>(band_smem + kBandStages * kBandStageBytes);
  const int lane = threadIdx.x & 31;
  // the warp's index through a shuffle: ptxas then knows that everything derived from it (rows,
  // presence masks) is warp-uniform and emits plain uniform branches
  const int warp = __shfl_sync(0xffffffffu, int(threadIdx.x >> 5), 0);
  const float4 *hv = reinterpret_cast<const float4 *>(h) + lane;      // row r -> hv[r * 32]
  float4 *zv = reinterpret_cast<float4 *>(z) + lane;
  float4 t[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) t[k] = reinterpret_cast<const float4 *>(table + k * kHidden)[lane];
  const int tiles = (n + kBandTile - 1) / kBandTile;
  auto tile_row0 = [&](int j) {                    // first row of this block's j-th tile, or -1
    const int v = int(blockIdx.x) + j * int(gridDim.x);
    return v < tiles ? (tiles - 1 - v) * kBandTile : -1;              // descending (L2 hand-over)
  };
  auto issue = [&](int j) {                        // one thread: tile j -> stage j % 3
    const int r0 = tile_row0(j);
    if (r0 < 0) return;
    const int lo = max(r0 - 2, 0), hi = min(r0 + kBandTile + 2, n);
    const uint32_t bytes = uint32_t(hi - lo) * (kHidden * 4);
    uint64_t *bar = &full[j % kBandStages];
    mbar_arrive_expect_tx(bar, bytes);
    bulk_g2s(band_smem + (j % kBandStages) * kBandStageBytes + (lo - (r0 - 2)) * (kHidden * 4),
             h + int64_t(lo) * kHidden, bytes, bar);
  };
  auto my_desc = [&](int r0) {                     // lanes 0-7: the descriptors of the warp's rows
    const int i = r0 + warp * 8 + lane;
    return (r0 >= 0 && lane < 8 && i < n) ? desc[i] : 0u;
  };
  auto prefetch_mates = [&](uint32_t d) {          // lanes 0-7: partner row of my row into L2
    if (d & kPair) {
      const char *p = reinterpret_cast<const char *>(h) + (int64_t((d >> kPartnerShift) & kPartnerMask) << 9);
#pragma unroll
      for (int q = 0; q < 4; ++q) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + q * 128));
    }
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kBandStages; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kBandStages; ++s) issue(s);
  }
  uint32_t mine = my_desc(tile_row0(0));
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int j = 0;; ++j) {
    const int r0 = tile_row0(j);
    if (r0 < 0) break;
    const int first = r0 + warp * 8;                                   // the warp's rows: first .. first + 7
    const int rows = min(n - first, 8);                                // <= 0: nothing to do in this tile
    const uint32_t m_prev = __ballot_sync(0xffffffffu, mine & kPrev),
                   m_next = __ballot_sync(0xffffffffu, mine & kNext),
                   m_pair = __ballot_sync(0xffffffffu, mine & kPair),
                   m_rev = __ballot_sync(0xffffffffu, mine & kPairRev),
                   m_prev2 = __ballot_sync(0xffffffffu, mine & kPrev2),
                   m_next2 = __ballot_sync(0xffffffffu, mine & kNext2);
    float4 mate[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const uint32_t d = __shfl_sync(0xffffffffu, mine, q);
      mate[q] = ((m_pair >> q) & 1u)
                    ? __ldg(hv + int64_t((d >> kPartnerShift) & kPartnerMask) * 32) : zero;
    }
    const uint32_t next_mine = my_desc(tile_row0(j + 1));
    prefetch_mates(next_mine);
    mbar_wait(&full[j % kBandStages], uint32_t(j / kBandStages) & 1u);
    // stage row s holds h row r0 - 2 + s; the warp's row q is stage row warp * 8 + q + 2
    const float4 *sv = reinterpret_cast<const float4 *>(band_smem + (j % kBandStages) * kBandStageBytes) +
                       warp * 8 * 32 + lane;
    float4 w[5];
#pragma unroll
    for (int s = 0; s < 4; ++s) w[s] = sv[s * 32];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (q >= rows) break;                                            // warp-uniform
      w[(q + 4) % 5] = sv[(q + 4) * 32];
      const float4 prev2 = w[q % 5], prev = w[(q + 1) % 5], self = w[(q + 2) % 5],
                   next = w[(q + 3) % 5], next2 = w[(q + 4) % 5];
      float4 acc = zero;
      if ((m_prev >> q) & 1u) band_add(acc, prev, t[0]);
      if ((m_next >> q) & 1u) band_add(acc, next, t[1]);
      if ((m_pair >> q) & 1u) band_add(acc, mate[q], ((m_rev >> q) & 1u) ? t[3] : t[2]);
      if ((m_prev2 >> q) & 1u) band_add(acc, prev2, t[4]);
      if ((m_next2 >> q) & 1u) band_add(acc, next2, t[5]);
      zv[int64_t(first + q) * 32] = make_float4(fmaf(eps1, self.x, acc.x), fmaf(eps1, self.y, acc.y),
                                                fmaf(eps1, self.z, acc.z), fmaf(eps1, self.w, acc.w));
    }
    mine = next_mine;
    __syncthreads();                                                   // every warp is done with the stage
    if (threadIdx.x == 0) issue(j + kBandStages);
  }
}

// ---------------------------------------------------------------------------
// SIMT MLP.  One warp owns 8 node rows end to end (both GEMMs, LayerNorm or
// L2 norm), so nothing but weights is shared between warps and only
// __syncwarp is needed.  Stage 1: lane owns HID/32 hidden columns of its 8
// rows; stage 2: lane owns 4 output columns.  Weights are read as [k][n]
// rows (coalesced 128-bit loads, L1/L2 resident: 256 KB per layer).
//   MODE 0:  out = res + LayerNorm(W2 relu(W1 a + b1) + b2) * g + b
//   MODE 1:  y = W2 relu(W1 a + b1) + b2 ; out[out_row] = y / max(|y|, 1e-12)
// ---------------------------------------------------------------------------
constexpr int kRowsPerWarp = 8;
constexpr int kMlpWarps = 8;

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

template <typename TIn, typename TOut, int HID, int MODE, bool ROUND_HIDDEN>
__global__ void __launch_bounds__(kMlpWarps * 32)
mlp_simt_kernel(const TIn *__restrict__ a_in, const TIn *__restrict__ res,
                const float *__restrict__ w1t, const float *__restrict__ b1,
                const float *__restrict__ w2t, const float *__restrict__ b2,
                const float *__restrict__ ln_g, const float *__restrict__ ln_b,
                const int32_t *__restrict__ out_row, int64_t n, TOut *__restrict__ out) {
  constexpr int C1 = HID / 32;  // hidden columns per lane
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *a_s = smem + warp * (kRowsPerWarp * (kHidden + HID));  // [8][128]
  float *h_s = a_s + kRowsPerWarp * kHidden;                    // [8][HID]
  const int64_t tiles = (n + kRowsPerWarp - 1) / kRowsPerWarp;
  for (int64_t tile = int64_t(blockIdx.x) * kMlpWarps + warp; tile < tiles;
       tile += int64_t(gridDim.x) * kMlpWarps) {
    const int64_t row0 = tile * kRowsPerWarp;
    // stage the 8 input rows (fp32 in shared memory)
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; ++r) {
      const int64_t row = row0 + r;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int col = lane + 32 * c;
        a_s[r * kHidden + col] = row < n ? to_f32<TIn>(a_in[row * kHidden + col]) : 0.f;
      }
    }
    __syncwarp();
    // ---- GEMM 1: hid[r][lane*C1 + c] -------------------------------------
    float acc1[kRowsPerWarp][C1];
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; ++r)
#pragma unroll
      for (int c = 0; c < C1; ++c) acc1[r][c] = b1[lane * C1 + c];
    for (int k = 0; k < kHidden; k += 4) {
      float4 av[kRowsPerWarp];
#pragma unroll
      for (int r = 0; r < kRowsPerWarp; ++r)
        av[r] = *reinterpret_cast<const float4 *>(a_s + r * kHidden + k);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        float w[C1];
        const float4 *wp = reinterpret_cast<const float4 *>(w1t + (k + kk) * HID + lane * C1);
#pragma unroll
        for (int c4 = 0; c4 < C1 / 4; ++c4) {
          float4 t = __ldg(wp + c4);
          w[4 * c4] = t.x; w[4 * c4 + 1] = t.y; w[4 * c4 + 2] = t.z; w[4 * c4 + 3] = t.w;
        }
#pragma unroll
        for (int r = 0; r < kRowsPerWarp; ++r) {
          const float a = kk == 0 ? av[r].x : kk == 1 ? av[r].y : kk == 2 ? av[r].z : av[r].w;
#pragma unroll
          for (int c = 0; c < C1; ++c) acc1[r][c] = fmaf(a, w[c], acc1[r][c]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; ++r)
#pragma unroll
      for (int c = 0; c < C1; ++c) {
        float v = fmaxf(acc1[r][c], 0.f);
        if (ROUND_HIDDEN) v = __half2float(__float2half_rn(v));
        h_s[r * HID + lane * C1 + c] = v;
      }
    __syncwarp();
    // ---- GEMM 2: u[r][lane*4 + c] -----------------------------------------
    float acc2[kRowsPerWarp][4];
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc2[r][c] = b2[lane * 4 + c];
    for (int k = 0; k < HID; k += 4) {
      float4 hv[kRowsPerWarp];
#pragma unroll
      for (int r = 0; r < kRowsPerWarp; ++r)
        hv[r] = *reinterpret_cast<const float4 *>(h_s + r * HID + k);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 w = __ldg(reinterpret_cast<const float4 *>(w2t + (k + kk) * kHidden + lane * 4));
#pragma unroll
        for (int r = 0; r < kRowsPerWarp; ++r) {
          const float a = kk == 0 ? hv[r].x : kk == 1 ? hv[r].y : kk == 2 ? hv[r].z : hv[r].w;
          acc2[r][0] = fmaf(a, w.x, acc2[r][0]);
          acc2[r][1] = fmaf(a, w.y, acc2[r][1]);
          acc2[r][2] = fmaf(a, w.z, acc2[r][2]);
          acc2[r][3] = fmaf(a, w.w, acc2[r][3]);
        }
      }
    }
    // ---- epilogue: a row's 128 values live in this warp (4 per lane) -------
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; ++r) {
      const int64_t row = row0 + r;
      if (MODE == 0) {
        float s = acc2[r][0] + acc2[r][1] + acc2[r][2] + acc2[r][3];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        const float mean = s * (1.f / kHidden);
        float q = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float dlt = acc2[r][c] - mean;
          q = fmaf(dlt, dlt, q);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) q += __shfl_xor_sync(0xffffffffu, q, d);
        const float rstd = rsqrtf(q * (1.f / kHidden) + 1e-5f);
        if (row < n) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int col = lane * 4 + c;
            const float u = (acc2[r][c] - mean) * rstd * ln_g[col] + ln_b[col];
            out[row * kHidden + col] =
                from_f32<TOut>(to_f32<TIn>(res[row * kHidden + col]) + u);
          }
        }
      } else {
        float q = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) q = fmaf(acc2[r][c], acc2[r][c], q);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) q += __shfl_xor_sync(0xffffffffu, q, d);
        const float inv = 1.f / fmaxf(sqrtf(q), 1e-12f);
        if (row < n) {
          const int64_t orow = out_row ? int64_t(out_row[row]) : row;
          if (orow >= 0) {
#pragma unroll
            for (int c = 0; c < 4; ++c)
              out[orow * kHidden + lane * 4 + c] = from_f32<TOut>(acc2[r][c] * inv);
          }
        }
      }
    }
    __syncwarp();
  }
}

template <typename TIn, typename TOut, int HID, int MODE, bool RH>
static int launch_mlp(const TIn *a, const TIn *res, const float *w1t, const float *b1,
                      const float *w2t, const float *b2, const float *g, const float *b,
                      const int32_t *out_row, int64_t n, TOut *out, cudaStream_t st) {
  auto kern = mlp_simt_kernel<TIn, TOut, HID, MODE, RH>;
  const size_t smem = size_t(kMlpWarps) * kRowsPerWarp * (kHidden + HID) * sizeof(float);
  GFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  const int64_t tiles = (n + kRowsPerWarp - 1) / kRowsPerWarp;
  int64_t blocks = (tiles + kMlpWarps - 1) / kMlpWarps;
  if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;
  kern<<<int(blocks), kMlpWarps * 32, smem, st>>>(a, res, w1t, b1, w2t, b2, g, b, out_row, n, out);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

// grid-stride kernels with a software pipeline: exactly the blocks that are
// resident at once (per_sm blocks of 256 threads per SM)
static inline int resident_grid(int64_t n, int per_sm) {
  int64_t b = (n + 15) / 16;
  int64_t cap = int64_t(kNumSMs) * per_sm;
  return int(b < 1 ? 1 : (b > cap ? cap : b));
}

static inline int row_grid(int64_t n) {
  int64_t b = (n + 15) / 16;
  int64_t cap = int64_t(kNumSMs) * 8;
  return int(b < 1 ? 1 : (b > cap ? cap : b));
}

// implemented in gfx_umma2.cu (general tcgen05 kernel) and gfx_umma4.cu (lean TMA kernel)
int umma_mlp_ln_residual(const gfx_model *m, int layer, const __half *z, const __half *h,
                         int64_t n, __half *h_out, cudaStream_t st);
int umma_head_l2norm(const gfx_model *m, const __half *h, const int32_t *out_row, int64_t n,
                     void *out, int out_dtype, cudaStream_t st);
int umma4_mlp_ln_residual(const gfx_model *m, int layer, const __half *z, const __half *h,
                          int64_t n, __half *h_out, cudaStream_t st);
// implemented in gfx_split9.cu: fp32 storage on the tensor cores (split-fp16 GEMMs)
int split9_mlp_ln_residual(const gfx_model *m, int layer, const float *z, const float *h, int64_t n,
                           float *h_out, cudaStream_t st);
int split9_head_l2norm(const gfx_model *m, const float *h, const int32_t *out_row, int64_t n, void *out,
                       int out_dtype, cudaStream_t st);
// implemented in gfx_head8.cu: fp16 in, fp16 out, identity row map
int head8_l2norm(const gfx_model *m, const __half *h, int64_t n, __half *out, cudaStream_t st);

}  // namespace gfx

namespace gfx {
int input8_linear(const gfx_model *m, const float *x, int64_t n, __half *h, cudaStream_t st);   // gfx_input8.cu
}

using namespace gfx;

extern "C" int gfx_input_linear(const gfx_model *m, const float *x, int64_t n, void *h, int dtype,
                                void *stream) {
  if (!m) return fail(GFX_ERR_ARGUMENT, "gfx_input_linear: null model");
  if (n <= 0) return GFX_OK;
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_INPUT, st, 1);
  if (dtype != GFX_F16 && dtype != GFX_F32)
    return fail(GFX_ERR_ARGUMENT, "gfx_input_linear: unknown dtype");
  // nodes before the first 16-byte aligned feature row (at most 3) take the
  // scalar kernel, the rest the vectorised one
  int64_t lead = 0;
  while (lead < n && lead < 4 && (reinterpret_cast<uintptr_t>(x + lead * kFeat) & 15)) ++lead;
  if (lead == 4) lead = n;                          // x is not even 4-byte aligned: scalar only
  const int64_t rest = n - lead;
  if (dtype == GFX_F16) {
    __half *hh = static_cast<__half *>(h);
    // the tensor-core kernel (gfx_input8.cu) when it applies, else the SIMT kernels
    const int rc = input8_linear(m, x, n, hh, st);
    if (rc != GFX_ERR_UNSUPPORTED) return rc;
    if (lead) input_linear_kernel<__half><<<row_grid(lead), 256, 0, st>>>(x, m->w_in[1], m->b_in, lead, hh);
    if (rest)
      input_linear4_kernel<__half><<<row_grid((rest + 3) / 4), 256, 0, st>>>(
          x + lead * kFeat, m->w_in[1], m->b_in, rest, hh + lead * kHidden);
  } else {
    float *hf = static_cast<float *>(h);
    if (lead) input_linear_kernel<float><<<row_grid(lead), 256, 0, st>>>(x, m->w_in[0], m->b_in, lead, hf);
    if (rest)
      input_linear4_kernel<float><<<row_grid((rest + 3) / 4), 256, 0, st>>>(
          x + lead * kFeat, m->w_in[0], m->b_in, rest, hf + lead * kHidden);
  }
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

extern "C" int gfx_aggregate(const gfx_model *m, int layer, const void *h, const int32_t *row_ptr,
                             const int32_t *col_src, const uint8_t *col_type, int64_t n, void *z,
                             int dtype, void *stream) {
  if (!m || layer < 0 || layer >= m->layers)
    return fail(GFX_ERR_ARGUMENT, "gfx_aggregate: bad model or layer");
  if (n <= 0) return GFX_OK;
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_AGGREGATE, st, 1);
  const size_t toff = size_t(layer) * m->edge_dim * kHidden;
  if (dtype == GFX_F16) {
    if (n <= (int64_t(1) << kSrcBits)) {
      int64_t b = (n + 31) / 32;
      const int grid = int(b > 4 * kNumSMs ? 4 * kNumSMs : b);
      aggregate_f16_q_kernel<<<grid, 256, 0, st>>>(
          static_cast<const __half *>(h), row_ptr, col_src, col_type, m->table16 + toff,
          m->edge_dim, m->eps1[layer], n, static_cast<__half *>(z));
    } else {
      aggregate_f16_kernel<<<resident_grid(n, 4), 256, 0, st>>>(
          static_cast<const __half *>(h), row_ptr, col_src, col_type, m->table16 + toff,
          m->edge_dim, m->eps1[layer], n, static_cast<__half *>(z));
    }
  } else if (dtype == GFX_F32) {
    if (n <= (int64_t(1) << kSrcBits)) {
      int64_t b = (n + 15) / 16;
      const int grid = int(b > 2 * kNumSMs ? 2 * kNumSMs : b);
      aggregate_f32_h_kernel<<<grid, 256, 0, st>>>(
          static_cast<const float *>(h), row_ptr, col_src, col_type, m->table[0] + toff,
          m->edge_dim, m->eps1[layer], n, static_cast<float *>(z), nullptr);
    } else {
      aggregate_kernel<float><<<row_grid(n), 256, 0, st>>>(
          static_cast<const float *>(h), row_ptr, col_src, col_type, m->table[0] + toff,
          m->edge_dim, m->eps1[layer], n, static_cast<float *>(z));
    }
  } else
    return fail(GFX_ERR_ARGUMENT, "gfx_aggregate: unknown dtype");
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

extern "C" int gfx_aggregate_banded(const gfx_model *m, int layer, const void *h, const uint32_t *desc,
                                    const int32_t *needs_csr, const int32_t *row_ptr,
                                    const int32_t *col_src, const uint8_t *col_type, int64_t n,
                                    void *z, int dtype, void *stream) {
  if (!m || layer < 0 || layer >= m->layers)
    return fail(GFX_ERR_ARGUMENT, "gfx_aggregate_banded: bad model or layer");
  if (dtype != GFX_F32)
    return fail(GFX_ERR_UNSUPPORTED, "gfx_aggregate_banded: fp32 storage only (the fp16 model has "
                                     "gfx_layer_fused_banded)");
  if (m->edge_dim < 6 || n > (int64_t(1) << rowdesc::kPartnerBits))
    return fail(GFX_ERR_UNSUPPORTED, "gfx_aggregate_banded: needs >= 6 edge types and <= 2^25 nodes");
  if (n <= 0) return GFX_OK;
  if (!desc || !needs_csr) return fail(GFX_ERR_ARGUMENT, "gfx_aggregate_banded: null descriptors or flag");
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_AGGREGATE, st, 2);
  const size_t toff = size_t(layer) * m->edge_dim * kHidden;
  {   // every row banded (*needs_csr == 0): the tile kernel; two blocks of eight warps per SM
    // per launch, not once per process: the attribute belongs to the current device
    GFX_CUDA(cudaFuncSetAttribute(aggregate_f32_band_kernel,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, kBandSmemBytes));
    const int64_t tiles = (n + kBandTile - 1) / kBandTile;
    const int grid = int(tiles > 2 * kNumSMs ? 2 * kNumSMs : tiles);
    aggregate_f32_band_kernel<<<grid, 256, kBandSmemBytes, st>>>(
        static_cast<const float *>(h), desc, needs_csr, m->table[0] + toff, m->eps1[layer], int(n),
        static_cast<float *>(z));
  }
  {   // some row GENERIC (*needs_csr != 0): the CSR kernel (gfx_csr_build_if built the arrays)
    int64_t b = (n + 15) / 16;
    const int grid = int(b > 2 * kNumSMs ? 2 * kNumSMs : b);
    aggregate_f32_h_kernel<<<grid, 256, 0, st>>>(
        static_cast<const float *>(h), row_ptr, col_src, col_type, m->table[0] + toff, m->edge_dim,
        m->eps1[layer], n, static_cast<float *>(z), needs_csr);
  }
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

extern "C" int gfx_mlp_ln_residual(const gfx_model *m, int layer, const void *z, const void *h,
                                   int64_t n, void *h_out, int dtype, int impl, void *stream) {
  if (!m || layer < 0 || layer >= m->layers)
    return fail(GFX_ERR_ARGUMENT, "gfx_mlp_ln_residual: bad model or layer");
  if (n <= 0) return GFX_OK;
  cudaStream_t st = as_stream(stream);
  const int H = kHidden, M = kMlpHidden;
  StageScope scope(GFX_STAGE_MLP, st, 1);
  if (impl == GFX_IMPL_AUTO) impl = dtype == GFX_F16 ? GFX_IMPL_UMMA_LEAN : GFX_IMPL_SPLIT;
  if (impl == GFX_IMPL_SPLIT) {
    if (dtype != GFX_F32)
      return fail(GFX_ERR_UNSUPPORTED, "split-fp16 tcgen05 MLP is the GFX_F32 path");
    if (n >= (int64_t(1) << 31) - 256)
      return fail(GFX_ERR_ARGUMENT, "split-fp16 tcgen05 MLP: node count must fit int32");
    return split9_mlp_ln_residual(m, layer, static_cast<const float *>(z), static_cast<const float *>(h),
                                  n, static_cast<float *>(h_out), st);
  }
  if (impl == GFX_IMPL_UMMA || impl == GFX_IMPL_UMMA_LEAN) {
    if (dtype != GFX_F16)
      return fail(GFX_ERR_UNSUPPORTED, "tcgen05 MLP exists for GFX_F16 only");
    auto fn = impl == GFX_IMPL_UMMA_LEAN ? umma4_mlp_ln_residual : umma_mlp_ln_residual;
    return fn(m, layer, static_cast<const __half *>(z), static_cast<const __half *>(h), n,
              static_cast<__half *>(h_out), st);
  }
  if (impl != GFX_IMPL_SIMT)
    return fail(GFX_ERR_ARGUMENT, "gfx_mlp_ln_residual: unknown impl (0 auto, 1 SIMT, 2 tcgen05, 5 lean tcgen05, 8 split tcgen05)");
  const int q = dtype == GFX_F16 ? 1 : 0;
  const float *w1t = m->w1t[q] + size_t(layer) * H * M, *b1 = m->b1 + size_t(layer) * M;
  const float *w2t = m->w2t[q] + size_t(layer) * M * H, *b2 = m->b2 + size_t(layer) * H;
  const float *g = m->ln_g + size_t(layer) * H, *b = m->ln_b + size_t(layer) * H;
  if (dtype == GFX_F16)
    return launch_mlp<__half, __half, kMlpHidden, 0, true>(
        static_cast<const __half *>(z), static_cast<const __half *>(h), w1t, b1, w2t, b2, g, b,
        nullptr, n, static_cast<__half *>(h_out), st);
  if (dtype == GFX_F32)
    return launch_mlp<float, float, kMlpHidden, 0, false>(
        static_cast<const float *>(z), static_cast<const float *>(h), w1t, b1, w2t, b2, g, b,
        nullptr, n, static_cast<float *>(h_out), st);
  return fail(GFX_ERR_ARGUMENT, "gfx_mlp_ln_residual: unknown dtype");
}

extern "C" int gfx_head_l2norm(const gfx_model *m, const void *h, const int32_t *out_row,
                               int64_t n, void *out, int dtype, int out_dtype, int impl,
                               void *stream) {
  if (!m) return fail(GFX_ERR_ARGUMENT, "gfx_head_l2norm: null model");
  if (n <= 0) return GFX_OK;
  if (out_dtype != GFX_F16 && out_dtype != GFX_F32)
    return fail(GFX_ERR_ARGUMENT, "gfx_head_l2norm: unknown out_dtype");
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_HEAD, st, 1);
  // the common case -- fp16 model, fp16 embeddings, every node a core node -- has its own kernel
  // with TMA tile I/O (gfx_head8.cu); GFX_IMPL_UMMA pins the general tcgen05 kernel (cross-check)
  if (impl == GFX_IMPL_AUTO && dtype == GFX_F16 && out_dtype == GFX_F16 && out_row == nullptr &&
      n <= (int64_t(1) << 30) && !((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(out)) & 15))
    return head8_l2norm(m, static_cast<const __half *>(h), n, static_cast<__half *>(out), st);
  if (impl == GFX_IMPL_AUTO) impl = dtype == GFX_F16 ? GFX_IMPL_UMMA : GFX_IMPL_SPLIT;
  if (impl == GFX_IMPL_SPLIT) {
    if (dtype != GFX_F32)
      return fail(GFX_ERR_UNSUPPORTED, "split-fp16 tcgen05 head is the GFX_F32 path");
    if (n >= (int64_t(1) << 31) - 256)
      return fail(GFX_ERR_ARGUMENT, "split-fp16 tcgen05 head: node count must fit int32");
    return split9_head_l2norm(m, static_cast<const float *>(h), out_row, n, out, out_dtype, st);
  }
  if (impl == GFX_IMPL_UMMA_LEAN) impl = GFX_IMPL_UMMA;  // head: general tcgen05 kernel
  if (impl == GFX_IMPL_UMMA) {
    if (dtype != GFX_F16)
      return fail(GFX_ERR_UNSUPPORTED, "tcgen05 head exists for GFX_F16 only");
    return umma_head_l2norm(m, static_cast<const __half *>(h), out_row, n, out, out_dtype, st);
  }
  if (impl != GFX_IMPL_SIMT)
    return fail(GFX_ERR_ARGUMENT, "gfx_head_l2norm: unknown impl (0 auto, 1 SIMT, 2 tcgen05, 8 split tcgen05)");
  const int q = dtype == GFX_F16 ? 1 : 0;
  if (dtype == GFX_F16 && out_dtype == GFX_F16)
    return launch_mlp<__half, __half, kHidden, 1, true>(
        static_cast<const __half *>(h), nullptr, m->wat[q], m->ba, m->wbt[q], m->bb, nullptr,
        nullptr, out_row, n, static_cast<__half *>(out), st);
  if (dtype == GFX_F16 && out_dtype == GFX_F32)
    return launch_mlp<__half, float, kHidden, 1, true>(
        static_cast<const __half *>(h), nullptr, m->wat[q], m->ba, m->wbt[q], m->bb, nullptr,
        nullptr, out_row, n, static_cast<float *>(out), st);
  if (dtype == GFX_F32 && out_dtype == GFX_F16)
    return launch_mlp<float, __half, kHidden, 1, false>(
        static_cast<const float *>(h), nullptr, m->wat[q], m->ba, m->wbt[q], m->bb, nullptr,
        nullptr, out_row, n, static_cast<__half *>(out), st);
  if (dtype == GFX_F32 && out_dtype == GFX_F32)
    return launch_mlp<float, float, kHidden, 1, false>(
        static_cast<const float *>(h), nullptr, m->wat[q], m->ba, m->wbt[q], m->bb, nullptr,
        nullptr, out_row, n, static_cast<float *>(out), st);
  return fail(GFX_ERR_ARGUMENT, "gfx_head_l2norm: unknown dtype");
}
