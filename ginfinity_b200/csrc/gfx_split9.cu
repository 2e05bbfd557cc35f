// full_precision=True on the tensor cores: K2 (MLP + LayerNorm + residual) and K3 (head + L2
// normalise) for fp32 STORAGE (GFX_F32, reference api.py:110-112 without .half()) as split-fp16
// tcgen05 GEMMs on CTA pairs.
//
// Round 1 ran these two stages on CUDA cores (26-34 TFLOP/s, 41 M nt/s for the whole fp32
// encoder): 131,072 + 65,536 dense FLOP per nucleotide cannot come from the fp32 pipe at the rate
// the rest of the path runs.  tcgen05 has no fp32 input kind and kind::tf32 keeps 10 mantissa
// bits -- ~1e-3 per product, two orders of magnitude above this path's 2e-5 parity bound -- so
// every fp32 operand x is split into two fp16 numbers
//        x = hi + lo,   hi = fp16(x),   lo = fp16(x - hi)          (|x - hi - lo| <= 2^-22 |x|)
// and every product A B^T becomes three fp16 MMAs accumulated in fp32 in TMEM:
//        A B^T ~= Ahi Bhi^T + Alo Bhi^T + Ahi Blo^T                (the lo x lo term is below 2^-22).
// Values here are far inside fp16's range (|z| < 64, |w| < 8); lo parts of tiny values become
// fp16 subnormals, which bounds their ABSOLUTE error by 3e-8 -- nothing next to sums of O(1).
//
// One kernel, two modes.  Per CTA pair (tcgen05 cta_group::2, M = 256 over two 128-row tiles; each
// CTA holds half of the N rows of every weight image, hi and lo: 128 KB in layer mode):
//   converters (8 warps)  fp32 rows of the input (z, or h for the head) from global memory ->
//                         hi / lo fp16 tiles in shared memory (K-major, 128-byte swizzle)
//   MMA issuer            GEMM 1: three operand combinations x 8 K-steps into D1 (fp32, TMEM);
//                         GEMM 2: three combinations x N1/16 K-steps from TMEM operands into D2
//   epilogue A (4 warps)  D1 + b1 -> ReLU -> hi packed in place over D1, lo into its own columns
//   epilogue B (8 warps)  layer: D2 + b2 -> LayerNorm -> * g + b + residual (fp32, global) -> fp32
//                         head:  D2 + bb -> L2 normalise (1e-12 clamp) -> cast -> out[out_row[i]]
// TMEM (512 columns): D1 [0, N1) with the hi operand of GEMM 2 in place at [0, N1/2); D2
// [256, 384); the lo operand at [384, 384 + N1/2).
#include <cstdlib>

#include "gfx_common.cuh"
#include "gfx_pair.cuh"
#include "gfx_umma.cuh"
#include "gfx_layer_math.cuh"

namespace gfx {

using namespace ptx;

namespace v9 {

using lmath::f2_add;
using lmath::f2_fma;
using lmath::kKbBytes;
using lmath::lds_f2;
using lmath::named_bar_sync;
using lmath::pack2;
using lmath::relu_pack2;
using lmath::sts64;
using lmath::sts_f2;

constexpr int kTileM = 128;
constexpr int kTileBytes = 2 * kKbBytes;      // a [128 x 128] fp16 tile: two K blocks
constexpr uint32_t kTmemCols = 512, kD2Col = 256, kLoCol = 384;
constexpr int kEpiBWarp0 = 4, kEpiBWarps = 8, kConvWarp0 = 12, kConvWarps = 8, kMmaWarp = 20, kWarps = 24;
constexpr int kRowsPerWarp = kTileM / kConvWarps;

enum Bar {
  kBarWLocal = 0, kBarWReady, kBarA1Full, kBarA1Empty, kBarD1Full, kBarA2Full, kBarD2Full,
  kBarD2Empty, kNumBars
};

template <int N1>
struct Smem {
  static constexpr int w1_piece = (N1 / 2) * 128;                    // one K block of this CTA's W1 rows
  static constexpr int w1_bytes = 2 * w1_piece;                      // K = 128: two K blocks
  static constexpr int w2_piece = 64 * 128;                          // 64 rows x one K block
  static constexpr int w2_bytes = (N1 / 64) * w2_piece;              // K = N1
  static constexpr int off_w1h = 0;
  static constexpr int off_w1l = off_w1h + w1_bytes;
  static constexpr int off_w2h = off_w1l + w1_bytes;
  static constexpr int off_w2l = off_w2h + w2_bytes;
  static constexpr int off_ah = off_w2l + w2_bytes;                  // input tile, hi
  static constexpr int off_al = off_ah + kTileBytes;                 // input tile, lo
  static constexpr int off_x = off_al + kTileBytes;                  // float2 [2 halves][128 rows]
  static constexpr int off_bar = off_x + 2 * kTileM * 8;
  static constexpr int off_tmem = off_bar + kNumBars * 8;
  static constexpr int total = off_tmem + 8;
};
static_assert(Smem<256>::total <= 232448, "exceeds the 227 KB shared-memory limit of sm_100");

struct Consts {
  float b1[kMlpHidden];
  float b2[kHidden], g[kHidden], be[kHidden];
};

struct Args {
  const float *in;           // [n, 128] fp32: z (layer) or h (head)
  const float *res;          // [n, 128] fp32 residual (layer mode)
  void *out;                 // layer: fp32 [n, 128]; head: fp16 or fp32 [*, 128]
  const int32_t *out_row;    // head: row map (null = identity, < 0 = dropped)
  const __half *w1h, *w1l, *w2h, *w2l;   // K-major swizzled images (gfx_api.cu)
  int64_t n;
  int out_half;              // head: 1 = fp16 output
};

__device__ __forceinline__ void mbar_wait_s(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) __nanosleep(64);
}
__device__ __forceinline__ float2 unpack2(uint32_t h2) {
  return __half22float2(*reinterpret_cast<const __half2 *>(&h2));
}
// x -> (hi, lo) on a pair of values; `relu` folds max(x, 0) into the split
template <bool RELU>
__device__ __forceinline__ void split2(float2 x, uint32_t &hi, uint32_t &lo) {
  if (RELU) {
    x.x = fmaxf(x.x, 0.f);
    x.y = fmaxf(x.y, 0.f);
  }
  hi = pack2(x.x, x.y);
  const float2 back = unpack2(hi);
  lo = pack2(x.x - back.x, x.y - back.y);
}

// 256-bit global accesses (LDG.E.ENL2.256 / STG.E.ENL2.256 on sm_100).  Epilogue B holds one ROW
// per thread (the TMEM lane), so a warp's access touches 32 different 128-byte lines whatever its
// width: with 16 bytes per thread the residual reads and the output stores of a tile were 8,192
// L1 wavefronts (ncu: the LSU data pipe 79 % busy, the tensor pipe waiting behind it); 32 bytes
// per thread -- a whole sector -- halves the requests and the wavefronts.  32-byte aligned.
__device__ __forceinline__ void ldg256(const float *p, float *v) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void stg256(float *p, const float *v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]),
               "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ void stg256(void *p, const uint32_t *v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

template <int N1, bool HEAD>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kWarps * 32, 1)
split_kernel(const __grid_constant__ Consts c, const Args p) {
  using L = Smem<N1>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::off_bar);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::off_tmem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();

  if (warp == kMmaWarp) {
    tmem_alloc2(tmem_slot, kTmemCols);
  } else if (tid == 0) {
    mbar_init(bar + kBarWLocal, 1);
    mbar_init(bar + kBarWReady, 2);
    mbar_init(bar + kBarA1Full, 2 * kConvWarps);
    mbar_init(bar + kBarA1Empty, 1);
    mbar_init(bar + kBarD1Full, 1);
    mbar_init(bar + kBarA2Full, 8);
    mbar_init(bar + kBarD2Full, 1);
    mbar_init(bar + kBarD2Empty, 2 * kEpiBWarps);
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int64_t n = p.n;
  const int tiles = int((n + kTileM - 1) / kTileM);
  const int pairs = (tiles + 1) / 2;
  const int cluster_id = blockIdx.x >> 1, clusters = gridDim.x >> 1;
  auto leader = [&](int b) { return map_to_cta(smem_u32(bar + b), 0); };

  if (warp < kEpiBWarp0) {
    // ================= epilogue A: D1 + b1 -> ReLU -> (hi, lo) fp16 operands in TMEM ===========
    reg_dec<72>();
    const uint32_t trow = tmem + (uint32_t(warp * 32) << 16);
    const uint32_t a2f = leader(kBarA2Full);
    uint32_t it = 0;
    for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
      mbar_wait_s(bar + kBarD1Full, it & 1);
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < N1 / 32; ++q) {
        float v[32];
        tmem_ld32(trow + 32 * q, v);
        tmem_ld_wait();
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 t = f2_add(make_float2(v[2 * j], v[2 * j + 1]),
                                  make_float2(c.b1[32 * q + 2 * j], c.b1[32 * q + 2 * j + 1]));
          split2<true>(t, hi[j], lo[j]);
        }
        tmem_st16(trow + 16 * q, hi);                 // in place: below what has been read
        tmem_st16(trow + kLoCol + 16 * q, lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(a2f);
    }
  } else if (warp < kConvWarp0) {
    // ================= epilogue B ===============================================================
    reg_inc<96>();
    const int quad = warp & 3, half = (warp - kEpiBWarp0) >> 2;
    const int r = quad * 32 + lane;
    const uint32_t xme = smem_u32(smem + L::off_x) + uint32_t(half * kTileM + r) * 8u;
    const uint32_t xother = smem_u32(smem + L::off_x) + uint32_t((half ^ 1) * kTileM + r) * 8u;
    const uint32_t d2e = leader(kBarD2Empty);
    const uint32_t tcol = tmem + (uint32_t(quad * 32) << 16) + kD2Col + uint32_t(half) * 64u;
    uint32_t it = 0;
    for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
      const int64_t row = int64_t(2 * pair + int(rank)) * kTileM + r;
      mbar_wait_s(bar + kBarD2Full, it & 1);
      tc_fence_after();
      float t[64];
      tmem_ld32(tcol, t);
      tmem_ld32(tcol + 32, t + 32);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(d2e);           // the accumulator is in registers now
      float2 s1 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int col = half * 64 + 2 * j;
        const float2 v = f2_add(make_float2(t[2 * j], t[2 * j + 1]), make_float2(c.b2[col], c.b2[col + 1]));
        t[2 * j] = v.x;
        t[2 * j + 1] = v.y;
        s1 = f2_add(s1, v);
        s2 = f2_fma(v, v, s2);
      }
      sts_f2(xme, make_float2(s1.x + s1.y, s2.x + s2.y));
      named_bar_sync(1u + uint32_t(quad), 64);
      const float2 other = lds_f2(xother);
      named_bar_sync(1u + uint32_t(quad), 64);
      const float sum = (s1.x + s1.y) + other.x, sq = (s2.x + s2.y) + other.y;
      if (!HEAD) {
        // h_out = h + LayerNorm(t) * g + be            (_model.py:68-71, fp32)
        const float mean = sum * (1.f / kHidden);
        const float var = fmaxf(sq * (1.f / kHidden) - mean * mean, 0.f);
        const float rstd = rsqrtf(var + 1e-5f);
        const float nm = -mean * rstd;
        if (row < n) {
          const float *res = p.res + row * kHidden + half * 64;
          float *out = static_cast<float *>(p.out) + row * kHidden + half * 64;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float rr[8], o[8];
            ldg256(res + 8 * k, rr);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int col = half * 64 + 8 * k + e;
              o[e] = fmaf(fmaf(t[8 * k + e], rstd, nm), c.g[col], c.be[col]) + rr[e];
            }
            stg256(out + 8 * k, o);
          }
        }
      } else {
        // out[out_row[i]] = y / max(|y|, 1e-12), cast          (api.py:250-259)
        const float inv = 1.f / fmaxf(sqrtf(sq), 1e-12f);
        int64_t dst = row < n ? row : -1;
        if (dst >= 0 && p.out_row != nullptr) dst = p.out_row[row];
        if (dst >= 0) {
          if (p.out_half) {
            __half *out = static_cast<__half *>(p.out) + dst * kHidden + half * 64;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              uint32_t o[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) o[e] = pack2(t[16 * k + 2 * e] * inv, t[16 * k + 2 * e + 1] * inv);
              stg256(out + 16 * k, o);
            }
          } else {
            float *out = static_cast<float *>(p.out) + dst * kHidden + half * 64;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              float o[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) o[e] = t[8 * k + e] * inv;
              stg256(out + 8 * k, o);
            }
          }
        }
      }
    }
  } else if (warp < kMmaWarp) {
    // ================= converters: fp32 rows -> hi / lo fp16 operand tiles ======================
    reg_inc<88>();     // 128 x 72 + 256 x 96 + 256 x 88 + 128 x 40 = 61,440 = the launch allocation
    const int pw = warp - kConvWarp0;
    // this lane's 4 channels = 8 bytes of a row: 16-byte chunk lane / 2 of the 256-byte fp16 row
    const uint32_t kboff = uint32_t(lane >> 4) * kKbBytes;
    const uint32_t c8 = uint32_t(lane >> 1) & 7u, odd8 = uint32_t(lane & 1) * 8u;
    auto cell = [&](int rr) -> uint32_t {
      return kboff + uint32_t(rr) * 128u + (((c8 ^ uint32_t(rr)) & 7u) << 4) + odd8;
    };
    const uint32_t ahs = smem_u32(smem + L::off_ah), als = smem_u32(smem + L::off_al);
    const uint32_t a1f = leader(kBarA1Full);
    uint32_t it = 0;
    for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
      const int64_t row0 = int64_t(2 * pair + int(rank)) * kTileM + kRowsPerWarp * pw;
      float4 v[kRowsPerWarp / 2];
#pragma unroll 1
      for (int part = 0; part < 2; ++part) {
#pragma unroll
        for (int j = 0; j < kRowsPerWarp / 2; ++j) {     // 8 independent 512-byte row reads in flight
          const int64_t row = row0 + part * (kRowsPerWarp / 2) + j;
          v[j] = row < n ? __ldg(reinterpret_cast<const float4 *>(p.in + row * kHidden) + lane)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (part == 0) mbar_wait_s(bar + kBarA1Empty, (it & 1) ^ 1);     // the tile has been consumed
#pragma unroll
        for (int j = 0; j < kRowsPerWarp / 2; ++j) {
          uint2 hi, lo;
          split2<false>(make_float2(v[j].x, v[j].y), hi.x, lo.x);
          split2<false>(make_float2(v[j].z, v[j].w), hi.y, lo.y);
          const uint32_t off = cell(kRowsPerWarp * pw + part * (kRowsPerWarp / 2) + j);
          sts64(ahs + off, hi);
          sts64(als + off, lo);
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(a1f);
    }
  } else if (warp == kMmaWarp) {
    // ================= weights (both CTAs) + MMA issue (rank 0) =================================
    reg_dec<40>();
    if (lane == 0) {
      mbar_arrive_expect_tx(bar + kBarWLocal, 2 * L::w1_bytes + 2 * L::w2_bytes);
      for (int lo = 0; lo < 2; ++lo) {
        const uint8_t *w1g = reinterpret_cast<const uint8_t *>(lo ? p.w1l : p.w1h);
        const uint8_t *w2g = reinterpret_cast<const uint8_t *>(lo ? p.w2l : p.w2h);
        uint8_t *w1s = smem + (lo ? L::off_w1l : L::off_w1h), *w2s = smem + (lo ? L::off_w2l : L::off_w2h);
        // W1 image: [2 K blocks][N1 rows][128 B]; this CTA's rows [N1/2 rank, +N1/2) of each block
        for (int kb = 0; kb < 2; ++kb)
          for (int off = 0; off < L::w1_piece; off += 8192)
            bulk_g2s(w1s + kb * L::w1_piece + off,
                     w1g + kb * (N1 * 128) + (N1 / 2) * int(rank) * 128 + off, 8192, bar + kBarWLocal);
        // W2 image: [N1/64 K blocks][128 rows][128 B]; rows [64 rank, +64) of each block
        for (int kb = 0; kb < N1 / 64; ++kb)
          bulk_g2s(w2s + kb * L::w2_piece, w2g + kb * (kHidden * 128) + 64 * int(rank) * 128,
                   L::w2_piece, bar + kBarWLocal);
      }
      mbar_wait_parked(bar + kBarWLocal, 0);
      mbar_arrive_cluster(leader(kBarWReady));
    }
    __syncwarp();
    if (rank == 0) {
      // The whole warp runs the tile loop and waits; one elected lane issues, so that the MMA
      // operands are warp-uniform to the compiler and live in uniform registers (issued from
      // inside `if (lane == 0)` every tcgen05.mma came wrapped in an ELECT / R2UR.BROADCAST
      // loop: 11-13 instructions for each of this kernel's 72 MMAs per tile pair; DESIGN.md 9.1).
      mbar_wait_parked(bar + kBarWReady, 0);
      const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
      uint32_t elected;
      asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(elected));
      const bool issuer = elected != 0u;
      constexpr uint32_t idesc1 = idesc_f16(2 * kTileM, N1);
      constexpr uint32_t idesc2 = idesc_f16(2 * kTileM, kHidden);
      const uint64_t w1d[2] = {smem_desc_sw128(smem_u32(smem + L::off_w1h)), smem_desc_sw128(smem_u32(smem + L::off_w1l))};
      const uint64_t w2d[2] = {smem_desc_sw128(smem_u32(smem + L::off_w2h)), smem_desc_sw128(smem_u32(smem + L::off_w2l))};
      const uint64_t ad[2] = {smem_desc_sw128(smem_u32(smem + L::off_ah)), smem_desc_sw128(smem_u32(smem + L::off_al))};
      uint32_t it = 0;
      for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
        mbar_wait_parked(bar + kBarA1Full, it & 1);
        tc_fence_after();
        if (issuer) {
          // GEMM 1: hi x hi, lo x hi, hi x lo  (operand A index, operand B index)
#pragma unroll
          for (int combo = 0; combo < 3; ++combo) {
            const int ai = combo == 1 ? 1 : 0, bi = combo == 2 ? 1 : 0;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              const int kb = kk >> 2, k = kk & 3;
              mma2_f16_ss(tm, ad[ai] + uint64_t((kb * kKbBytes + k * 32) >> 4),
                          w1d[bi] + uint64_t((kb * L::w1_piece + k * 32) >> 4), idesc1,
                          (combo | kk) != 0);
            }
          }
          mma2_commit(bar + kBarD1Full);
          mma2_commit(bar + kBarA1Empty);
        }
        __syncwarp();
        mbar_wait_parked(bar + kBarA2Full, it & 1);
        mbar_wait_parked(bar + kBarD2Empty, (it & 1) ^ 1);
        tc_fence_after();
        if (issuer) {
#pragma unroll
          for (int combo = 0; combo < 3; ++combo) {
            const uint32_t a_tmem = tm + (combo == 1 ? kLoCol : 0u);
            const int bi = combo == 2 ? 1 : 0;
#pragma unroll
            for (int kk = 0; kk < N1 / 16; ++kk)
              mma2_f16_ts(tm + kD2Col, a_tmem + kk * 8,
                          w2d[bi] + uint64_t(((kk >> 2) * L::w2_piece + (kk & 3) * 32) >> 4), idesc2,
                          (combo | kk) != 0);
          }
          mma2_commit(bar + kBarD2Full);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else {
    reg_dec<40>();                                // spare warps of the utility warpgroup
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                             // the peer may still be arriving on our barriers
  if (warp == kMmaWarp) tmem_dealloc2(tmem, kTmemCols);
}

template <int N1, bool HEAD>
static int launch(const Consts &c, const Args &a, cudaStream_t st) {
  auto kernel = split_kernel<N1, HEAD>;
  constexpr int smem = Smem<N1>::total;
  GFX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int64_t tiles = (a.n + kTileM - 1) / kTileM;
  const int64_t pairs = (tiles + 1) / 2;
  int cap = 0;
  if (const int rc = resident_pairs<split_kernel<N1, HEAD>>(kWarps * 32, smem, &cap)) return rc;
  const int clusters = int(pairs < cap ? pairs : cap);
  kernel<<<2 * clusters, kWarps * 32, smem, st>>>(c, a);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

}  // namespace v9

// K2 for fp32 storage: h_out = h + LayerNorm(W2 relu(W1' z + b1') + b2), all arrays fp32 [n, 128]
int split9_mlp_ln_residual(const gfx_model *m, int layer, const float *z, const float *h, int64_t n,
                           float *h_out, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(h) |
       reinterpret_cast<uintptr_t>(h_out)) & 31)
    return fail(GFX_ERR_ARGUMENT, "split tcgen05 MLP: activation buffers must be 32-byte aligned");
  v9::Consts c{};
  const gfx_host_vectors &hv = m->host;
  for (int i = 0; i < kMlpHidden; ++i) c.b1[i] = hv.b1[size_t(layer) * kMlpHidden + i];
  for (int i = 0; i < kHidden; ++i) {
    c.b2[i] = hv.b2[size_t(layer) * kHidden + i];
    c.g[i] = hv.ln_g[size_t(layer) * kHidden + i];
    c.be[i] = hv.ln_b[size_t(layer) * kHidden + i];
  }
  const size_t wi = size_t(layer) * kMlpHidden * kHidden;
  v9::Args a{};
  a.in = z; a.res = h; a.out = h_out; a.n = n;
  a.w1h = m->w1_img + wi; a.w1l = m->w1_lo_img + wi;
  a.w2h = m->w2_img + wi; a.w2l = m->w2_lo_img + wi;
  return v9::launch<kMlpHidden, false>(c, a, st);
}

// K3 for fp32 storage: y = Wb relu(Wa h + ba) + bb; out[out_row[i]] = y_i / max(|y_i|, 1e-12)
int split9_head_l2norm(const gfx_model *m, const float *h, const int32_t *out_row, int64_t n, void *out,
                       int out_dtype, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(out)) & 31)
    return fail(GFX_ERR_ARGUMENT, "split tcgen05 head: buffers must be 32-byte aligned");
  v9::Consts c{};
  const gfx_host_vectors &hv = m->host;
  for (int i = 0; i < kHidden; ++i) {
    c.b1[i] = hv.ba[i];
    c.b2[i] = hv.bb[i];
  }
  v9::Args a{};
  a.in = h; a.out = out; a.out_row = out_row; a.n = n; a.out_half = out_dtype == GFX_F16 ? 1 : 0;
  a.w1h = m->wa_img; a.w1l = m->wa_lo_img; a.w2h = m->wb_img; a.w2l = m->wb_lo_img;
  return v9::launch<kHidden, true>(c, a, st);
}

}  // namespace gfx
