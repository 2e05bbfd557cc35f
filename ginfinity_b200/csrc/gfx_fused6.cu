// One GINE layer in one kernel on CTA PAIRS (tcgen05 cta_group::2): K1 (the
// aggregation) produces K2's GEMM-1 A operand in shared memory, so z never
// exists in HBM and h is read once and written once per layer.
//
//   h_out = h + LayerNorm(W2 relu(W1' z + b1') + b2),
//   z_i   = (1+eps) h_i + sum_{e: dst=i} relu(h[src_e] + table[type_e])
//
// Why pairs: gfx_fused5.cu (one CTA per SM) keeps 128 KB of weights resident
// and has 99 KB left, i.e. two 32 KB buffers that each have to be z tile,
// residual tile and output tile in turn; their life cycle, not the tensor
// pipe, set its pace (DESIGN.md section 9).  A CTA pair splits the B operands
// (each CTA holds the half of W1 / W2 that produces half of the N columns:
// 64 KB), runs M = 256 MMAs over both CTAs' 128-row tiles, and has 160 KB per
// CTA for data:
//   * 3 h-tile buffers (32 KB, TMA, 128-byte swizzle): the tile's own rows of
//     h serve (i) the producers' self rows and in-tile neighbour rows (~97 % of
//     the edges of RNA graphs stay inside a 128-row tile; the rest are read
//     from global memory / L2), (ii) epilogue B's residual, (iii) the output
//     staging for the TMA store -- loaded once, stored once;
//   * 2 z stages (32 KB, the UMMA K-major swizzled A operand of GEMM 1).
// TMEM (512 columns per CTA): D1 [0,256) fp32, overwritten IN PLACE by the
// fp16 hidden activation A2 [0,128) (epilogue A walks the columns upwards, so
// it only overwrites what it has already read), D2 double-buffered at
// [256,384) and [384,512).
//
// Warps (24; 80 registers per thread at launch, re-balanced with setmaxnreg: the producers get
// 104, the utility warpgroup 40), per CTA:
//    0-3   epilogue A   D1 -> + b1, ReLU, fp16 -> A2 (in place)
//    4-11  epilogue B   two groups of 4, alternating tiles: D2 -> + b2,
//                       LayerNorm (two passes over TMEM, full rows: no
//                       exchange between warps), + residual, in place in the
//                       h-tile buffer
//   12-19  producers    quarter-warp per node (as K1: shuffled edge fetch,
//                       branch-free missing edges), rows from the h-tile
//                       buffer, z row into the z stage; the CSR entries of the
//                       NEXT tile are fetched before the current one is summed
//   20     MMA issuer   (rank 0 of the pair issues for both CTAs; both fetch
//                       their halves of the weights)
//   21     h-tile loader (TMA)
//   22     output store  (TMA)
// Barriers that collect arrivals from both CTAs (z full, A2 full, D2 empty,
// weights ready) live in rank 0 and are reached with mapa + a cluster-scope
// arrive; completions of the MMAs are multicast to both CTAs by tcgen05.commit.
#include "gfx_common.cuh"
#include "gfx_tma.cuh"
#include "gfx_pair.cuh"
#include "gfx_umma.cuh"
#include "gfx_layer_math.cuh"

namespace gfx {

using namespace ptx;

namespace v6 {

constexpr int HID = kMlpHidden, H = HID / 2;
constexpr int kTileM = 128;
constexpr int kKbBytes = kTileM * 128;        // one K block of a tile: [128 x 64] fp16
constexpr int kTileBytes = 2 * kKbBytes;      // a whole [128 x 128] fp16 tile
constexpr int kStages = 2, kHBufs = 3;
constexpr int kWPiece = 64 * 128;             // 64 weight rows x 64 columns (one CTA's share)
constexpr int kTabRows = 11;                  // edge types 0..9 + the "no edge" row
constexpr uint32_t kTmemCols = 512, kD2Col = 256;
constexpr int kEpiBWarp0 = 4, kProdWarp0 = 12, kProdWarps = 8, kMmaWarp = 20, kLoadWarp = 21,
              kStoreWarp = 22, kWarps = 24;
constexpr int kQuarters = kProdWarps * 4;             // quarter-warps producing z rows
constexpr int kRowsPerQuarter = kTileM / kQuarters;   // rows of a tile per quarter-warp
static_assert(kRowsPerQuarter * kQuarters == kTileM, "tile rows must divide evenly");
constexpr int kSrcBits = 27;
constexpr uint32_t kSrcMask = (1u << kSrcBits) - 1u;
constexpr int kWin = 5;

enum Bar {
  kBarWLocal = 0, kBarWReady = 1, kBarHFull = 2, kBarHEmpty = 5, kBarOReady = 8, kBarA1Full = 11,
  kBarA1Empty = 13, kBarD1aFull = 15, kBarD1bFull = 16, kBarA2aFull = 17, kBarA2bFull = 18,
  kBarD2Full = 19, kBarD2Empty = 21, kNumBars = 23
};

struct Smem {
  static constexpr int off_w1 = 0;                                   // [kb 2] x 16 KB (128 rows)
  static constexpr int off_w2 = off_w1 + 4 * kWPiece;                // [kb 4] x 8 KB
  static constexpr int off_z = off_w2 + 4 * kWPiece;                 // 2 stages x 32 KB
  static constexpr int off_h = off_z + kStages * kTileBytes;         // 3 tiles x 32 KB
  static constexpr int off_tab = off_h + kHBufs * kTileBytes;        // fp16 [11][128]
  static constexpr int off_bar = off_tab + kTabRows * kHidden * 2;
  static constexpr int off_tmem = off_bar + kNumBars * 8;
  static constexpr int total = off_tmem + 8;
};
static_assert(Smem::total <= 232448, "exceeds the 227 KB shared-memory limit of sm_100");

struct alignas(64) Maps {
  CUtensorMap h, out;        // [n, 128] fp16, box 64 x 128, SWIZZLE_128B
};

using Consts = lmath::Consts;     // b1, b2, LayerNorm vectors as kernel parameters

struct Args {
  const __half *h;
  const int32_t *row_ptr, *col_src;
  const uint8_t *col_type;
  const __half *table16, *w1_img, *w2_img;
  int64_t n;
  int edge_dim;
  uint32_t eps1_h2;          // (1 + eps) rounded to fp16, in both halves of the word
};

// parked wait (suspend-time hint) on a local barrier
__device__ __forceinline__ void mbar_wait_c(uint64_t *bar, uint32_t parity) {
  mbar_wait_parked(bar, parity);
}
__device__ __forceinline__ void fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

__device__ __forceinline__ uint32_t relu_pack2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t hfma2_relu_add(uint32_t x, uint32_t t) {
  uint32_t r;
  asm volatile("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0x3c003c00u), "r"(t));
  return r;
}
__device__ __forceinline__ void add_pair(float &a0, float &a1, uint32_t m) {
  asm volatile("{\n.reg .b16 lo, hi;\nmov.b32 {lo, hi}, %2;\nadd.rn.f32.f16 %0, lo, %0;\n"
      "add.rn.f32.f16 %1, hi, %1;\n}"
      : "+f"(a0), "+f"(a1)
      : "r"(m));
}
// one message on 8 channels, in packed half like the reference's fp16 path (and gfx_fused8.cu):
// acc = half(acc + relu(half(x + t)))
__device__ __forceinline__ void add_message(uint32_t *acc, const uint4 &nb, const uint4 &tb) {
  acc[0] = lmath::h2_add(acc[0], lmath::h2_relu_add(nb.x, tb.x));
  acc[1] = lmath::h2_add(acc[1], lmath::h2_relu_add(nb.y, tb.y));
  acc[2] = lmath::h2_add(acc[2], lmath::h2_relu_add(nb.z, tb.z));
  acc[3] = lmath::h2_add(acc[3], lmath::h2_relu_add(nb.w, tb.w));
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(saddr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, const uint4 &v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}
// 16 bytes of a neighbour row: from the resident h tile when the source lies in this tile, else
// from global memory (L2).  One predicated instruction of each kind writing the SAME registers:
// written as an if/else, the compiler predicates both paths into separate registers and merges
// them with eight moves per row.
__device__ __forceinline__ uint4 ld_tile_or_global(uint32_t in_tile, uint32_t saddr, const uint4 *gptr) {
  uint4 v;
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "setp.ne.b32 q, %4, 0;\n"
      "@q ld.shared.v4.u32 {%0, %1, %2, %3}, [%5];\n"
      "@!q ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%6];\n"
      "}\n"
      : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
      : "r"(in_tile), "r"(saddr), "l"(gptr));
  return v;
}
// byte offset of 16-byte chunk `c8` (0..7) of row `r` inside one swizzled K block
__device__ __forceinline__ uint32_t sw_off(int r, int c8) {
  return uint32_t(r) * 128u + (uint32_t((c8 ^ r) & 7) << 4);
}

// D1[:, HALF*128 .. +128) -> bias + ReLU -> fp16 -> A2[:, HALF*64 .. +64), 32 columns at a time
template <int HALF>
__device__ __forceinline__ void epi_a(const Consts &c, uint32_t trow, uint64_t *bar, uint32_t ph,
                                      int lane, uint32_t leader_bar) {
  constexpr int col0 = HALF * H;
  mbar_wait_c(bar + (HALF ? kBarD1bFull : kBarD1aFull), ph);
  tc_fence_after();
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float v[32];
    tmem_ld32(trow + col0 + 32 * q, v);
    tmem_ld_wait();
    uint32_t pk[16];
#pragma unroll
    for (int j = 0; j < 16; ++j)
      pk[j] = relu_pack2(v[2 * j] + c.b1[col0 + 32 * q + 2 * j],
                         v[2 * j + 1] + c.b1[col0 + 32 * q + 2 * j + 1]);
    tmem_st16(trow + col0 / 2 + 16 * q, pk);
  }
  tmem_st_wait();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(leader_bar);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kWarps * 32, 1)
fused_pair_kernel(const __grid_constant__ Maps maps, const __grid_constant__ Consts c, const Args p) {
  using L = Smem;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *w1s = smem + L::off_w1, *w2s = smem + L::off_w2, *zs = smem + L::off_z;
  uint8_t *hs = smem + L::off_h;
  uint4 *tab = reinterpret_cast<uint4 *>(smem + L::off_tab);
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::off_bar);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::off_tmem);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  if (warp == kMmaWarp) {
    tmem_alloc2(tmem_slot, kTmemCols);
  } else if (tid == 0) {
    mbar_init(bar + kBarWLocal, 1);
    mbar_init(bar + kBarWReady, 2);
    for (int s = 0; s < kHBufs; ++s) {
      mbar_init(bar + kBarHFull + s, 1);
      mbar_init(bar + kBarHEmpty + s, 1);
      mbar_init(bar + kBarOReady + s, 4);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar + kBarA1Full + s, 2 * kProdWarps);
      mbar_init(bar + kBarA1Empty + s, 1);
      mbar_init(bar + kBarD2Full + s, 1);
      mbar_init(bar + kBarD2Empty + s, 8);
    }
    mbar_init(bar + kBarD1aFull, 1);
    mbar_init(bar + kBarD1bFull, 1);
    mbar_init(bar + kBarA2aFull, 8);
    mbar_init(bar + kBarA2bFull, 8);
    fence_mbar_init();
  }
  for (int i = tid; i < p.edge_dim * kHidden / 8; i += blockDim.x)
    tab[i] = reinterpret_cast<const uint4 *>(p.table16)[i];
  for (int i = tid; i < kHidden / 8; i += blockDim.x)               // the "no edge" row: -65504
    tab[p.edge_dim * kHidden / 8 + i] = make_uint4(0xFBFFFBFFu, 0xFBFFFBFFu, 0xFBFFFBFFu, 0xFBFFFBFFu);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                          // both CTAs' barriers exist before any remote arrive
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int n = int(p.n);
  const int tiles = (n + kTileM - 1) / kTileM;
  const int pairs = (tiles + 1) / 2;
  const int cluster_id = blockIdx.x >> 1, clusters = gridDim.x >> 1;
  // barriers of rank 0 that collect arrivals from both CTAs
  auto leader = [&](int b) { return map_to_cta(smem_u32(bar + b), 0); };

  if (warp < kEpiBWarp0) {
    // ================= epilogue A =================================================
    reg_dec<64>();
    const uint32_t trow = tmem + (uint32_t(warp * 32) << 16);
    const uint32_t a2a = leader(kBarA2aFull), a2b = leader(kBarA2bFull);
    uint32_t it = 0;
    for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
      epi_a<0>(c, trow, bar, it & 1, lane, a2a);
      epi_a<1>(c, trow, bar, it & 1, lane, a2b);
    }
  } else if (warp < kProdWarp0) {
    // ================= epilogue B (group g takes iterations it % 2 == g) ===========
    const int quad = warp & 3, g = (warp - kEpiBWarp0) >> 2;
    const uint32_t trow = tmem + (uint32_t(quad * 32) << 16) + kD2Col + uint32_t(g) * kHidden;
    const uint32_t d2e = leader(kBarD2Empty + g);
    const int r = quad * 32 + lane;
    uint32_t it = 0;
    for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
      if (int(it & 1) != g) continue;
      const uint32_t hb = it % kHBufs;
      mbar_wait_c(bar + kBarD2Full + g, (it >> 1) & 1);
      tc_fence_after();
      // the arithmetic of gfx_fused8.cu's epilogue B (gfx_layer_math.cuh), both column halves of
      // the row on this thread: same operations in the same order, same bits
      // (the column half is a run-time value here: two unrolled copies with their 384 constant
      // operands spill under this role's register limit)
      float2 part[2];
#pragma unroll 1
      for (int half = 0; half < 2; ++half) part[half] = lmath::epi_b_partial_rt(c, trow + 64 * half, half);
      const float2 lo = part[0], hi = part[1];
      const float sum = lo.x + hi.x, sq = lo.y + hi.y;
      const float mean = sum * (1.f / kHidden);
      const float var = fmaxf(sq * (1.f / kHidden) - mean * mean, 0.f);
      const float rstd = rsqrtf(var + 1e-5f);
      const float nm = -mean * rstd;
      mbar_wait_c(bar + kBarHFull + hb, (it / kHBufs) & 1);      // long complete: visibility only
      const uint32_t hrow = smem_u32(hs) + hb * kTileBytes;
#pragma unroll 1
      for (int half = 0; half < 2; ++half)
        lmath::epi_b_normalise_rt(c, trow + 64 * half, hrow, r, rstd, nm, half);
      tc_fence_before();                                         // D2 fully read
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(d2e);
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + kBarOReady + hb);
    }
  } else if (warp < kMmaWarp) {
    // ================= producers: aggregation into the z stage ======================
    reg_inc<104>();
    const int ptid = (warp - kProdWarp0) * 32 + lane;
    const int qid = ptid >> 3, sub = ptid & 7, qbase = lane & 24;
    const uint4 *hv = reinterpret_cast<const uint4 *>(p.h) + sub;     // row r -> hv[r*16], hv[r*16+8]
    const uint32_t tvs = smem_u32(tab) + uint32_t(sub) * 16u;          // type t -> tvs + t*256 (+128)
    const uint32_t a1f[2] = {leader(kBarA1Full), leader(kBarA1Full + 1)};

    // This quarter-warp owns rows qid + 32 k (k = 0..3) of every tile of its CTA: a sequence of
    // "row steps" j (tile iteration j / 4, row group j % 4).  The CSR entries travel through a
    // register pipeline so that no load is consumed near the step that issues it: row_ptr
    // three steps ahead (A), this lane's edge (source, type) two steps ahead (B1 -> B0),
    // packed and used now.
    const int my_iters = cluster_id < pairs ? (pairs - cluster_id + clusters - 1) / clusters : 0;
    const int steps = kRowsPerQuarter * my_iters;
    auto row_of = [&](int j) {
      return (2 * (cluster_id + (j / kRowsPerQuarter) * clusters) + int(rank)) * kTileM + qid +
             kQuarters * (j % kRowsPerQuarter);
    };
    int begA = 0, endA = 0, srcB0 = 0, typB0 = 0, srcB1 = 0, typB1 = 0;
    auto load_a = [&](int j) {
      begA = endA = 0;
      if (j < steps) {
        const int row = row_of(j);
        if (row < n) {
          begA = p.row_ptr[row];
          endA = p.row_ptr[row + 1];
        }
      }
    };
    auto load_b = [&](int j, int &src, int &typ) {       // consumes A
      const int row = j < steps ? row_of(j) : 0;
      src = row < n ? row : 0;                           // no edge: the node itself, "none" type
      typ = p.edge_dim;
      if (begA + sub < endA) {
        src = p.col_src[begA + sub];
        typ = p.col_type[begA + sub];
      }
    };
    load_a(0);
    load_b(0, srcB0, typB0);
    load_a(1);
    load_b(1, srcB1, typB1);
    load_a(2);
#pragma unroll 1
    for (int j = 0; j < steps; ++j) {
      const uint32_t it = uint32_t(j) / kRowsPerQuarter;
      const int k = j % kRowsPerQuarter;
      const uint32_t s = it & 1, hb = it % kHBufs;
      const int row0 = (2 * (cluster_id + int(it) * clusters) + int(rank)) * kTileM;
      const uint32_t pk = (uint32_t(srcB0) & kSrcMask) | (uint32_t(typB0) << kSrcBits);
      srcB0 = srcB1;
      typB0 = typB1;
      load_b(j + 2, srcB1, typB1);
      load_a(j + 3);
      const uint32_t hbase = smem_u32(hs) + hb * kTileBytes;
      const uint32_t zbase = smem_u32(zs) + s * kTileBytes;
      if (k == 0) {
        mbar_wait_c(bar + kBarHFull + hb, (it / kHBufs) & 1);
        mbar_wait_c(bar + kBarA1Empty + s, ((it >> 1) & 1) ^ 1);
      }
      const int lr = qid + kQuarters * k;
      uint32_t acc[8];                 // 16 channels as 8 half pairs (+0)
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) acc[ch] = 0u;
      // Half a row (16 bytes per lane) ahead: the next half row is requested before the current
      // one is summed.  The asm statements are volatile, so this order is the order of the
      // machine code; left to itself the compiler hoists all ten row loads and spills.
      struct Edge {
        uint32_t in_tile, a, t;        // smem address of the row chunk, table address
        const uint4 *gp;
      };
      auto edge = [&](int u) {
        const uint32_t e = __shfl_sync(0xffffffffu, pk, qbase + u);
        const int src = int(e & kSrcMask);
        const uint32_t local = uint32_t(src - row0);
        Edge x;
        x.in_tile = local < uint32_t(kTileM) ? 1u : 0u;
        x.a = hbase + sw_off(int(local), sub);
        x.gp = hv + int64_t(src) * 16;
        x.t = tvs + (e >> kSrcBits) * 256u;
        return x;
      };
      Edge cur = edge(0);
      uint4 d0 = ld_tile_or_global(cur.in_tile, cur.a, cur.gp);
#pragma unroll
      for (int u = 0; u < kWin; ++u) {
        const uint4 d1 = ld_tile_or_global(cur.in_tile, cur.a + kKbBytes, cur.gp + 8);
        add_message(acc, d0, lds128(cur.t));
        const uint32_t t1 = cur.t + 128u;
        if (u + 1 < kWin) {
          cur = edge(u + 1);
          d0 = ld_tile_or_global(cur.in_tile, cur.a, cur.gp);
        }
        add_message(acc + 4, d1, lds128(t1));
      }
      // rare: rows longer than the window (lane kWin of the quarter holds edge kWin, if any)
      if ((__shfl_sync(0xffffffffu, pk, qbase + kWin) >> kSrcBits) != uint32_t(p.edge_dim)) {
        const int beg = p.row_ptr[row0 + lr], end = p.row_ptr[row0 + lr + 1];
        for (int eidx = beg + kWin; eidx < end; ++eidx) {
          const int src = p.col_src[eidx];
          const uint32_t t = tvs + uint32_t(p.col_type[eidx]) * 256u;
          add_message(acc, hv[int64_t(src) * 16], lds128(t));
          add_message(acc + 4, hv[int64_t(src) * 16 + 8], lds128(t + 128u));
        }
      }
      uint4 o0 = make_uint4(0, 0, 0, 0), o1 = make_uint4(0, 0, 0, 0);
      const uint32_t so = sw_off(lr, sub);
      if (row0 + lr < n) {
        const uint4 self0 = lds128(hbase + so), self1 = lds128(hbase + so + kKbBytes);
        const uint32_t e1 = p.eps1_h2;
        o0 = make_uint4(lmath::h2_fma(e1, self0.x, acc[0]), lmath::h2_fma(e1, self0.y, acc[1]),
                        lmath::h2_fma(e1, self0.z, acc[2]), lmath::h2_fma(e1, self0.w, acc[3]));
        o1 = make_uint4(lmath::h2_fma(e1, self1.x, acc[4]), lmath::h2_fma(e1, self1.y, acc[5]),
                        lmath::h2_fma(e1, self1.z, acc[6]), lmath::h2_fma(e1, self1.w, acc[7]));
      }
      sts128(zbase + so, o0);
      sts128(zbase + so + kKbBytes, o1);
      if (k == kRowsPerQuarter - 1) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(a1f[s]);
      }
    }
  } else if (warp == kMmaWarp) {
    // ================= weights (both CTAs) + MMA issue (rank 0) ======================
    reg_dec<40>();
    if (lane == 0) {
      mbar_arrive_expect_tx(bar + kBarWLocal, 8 * kWPiece);
      const uint8_t *w1g = reinterpret_cast<const uint8_t *>(p.w1_img);
      const uint8_t *w2g = reinterpret_cast<const uint8_t *>(p.w2_img);
      // Each CTA supplies W1' rows [128 rank, +128) of every K block (two 8 KB pieces, contiguous:
      // one B operand of an N = 256 MMA).  In pair mode an MMA costs ~128 cycles whether N is 128
      // or 256 (measured with gfx_umma7.cu), so GEMM 1 runs as 8 MMAs of N = 256, not 16 of N = 128.
      for (int kb = 0; kb < 2; ++kb)
        for (int half = 0; half < 2; ++half)
          bulk_g2s(w1s + (kb * 2 + half) * kWPiece,
                   w1g + kb * (HID * 128) + (H * int(rank) + 64 * half) * 128, kWPiece,
                   bar + kBarWLocal);
      for (int kb = 0; kb < 4; ++kb)              // rows [64 rank, +64) of K block kb
        bulk_g2s(w2s + kb * kWPiece, w2g + kb * (kHidden * 128) + 64 * int(rank) * 128, kWPiece,
                 bar + kBarWLocal);
      mbar_wait_parked(bar + kBarWLocal, 0);
      mbar_arrive_cluster(leader(kBarWReady));
    }
    __syncwarp();
    if (rank == 0) {
      // the whole warp runs the tile loop and waits, one elected lane issues: MMA operands in
      // uniform registers instead of an ELECT / R2UR.BROADCAST loop around every tcgen05.mma
      // (gfx_fused8.cu, DESIGN.md section 9.1)
      mbar_wait_c(bar + kBarWReady, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
      uint32_t elected;
      asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(elected));
      const bool issuer = elected != 0u;
      {
        constexpr uint32_t idesc = idesc_f16(2 * kTileM, H);     // M = 256 over the pair, N = 128
        const uint32_t w1a = smem_u32(w1s), w2a = smem_u32(w2s);
        uint32_t it = 0;
        for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
          const uint32_t s = it & 1, g = it & 1, ph2 = (it >> 1) & 1, ph = it & 1;
          const uint32_t za = smem_u32(zs) + s * kTileBytes;
          mbar_wait_c(bar + kBarA1Full + s, ph2);
          tc_fence_after();
          if (issuer) {
            constexpr uint32_t idesc_w = idesc_f16(2 * kTileM, HID);   // GEMM 1: N = 256
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              const int kb = kk >> 2, k = kk & 3;
              const uint64_t da = smem_desc_sw128(za + kb * kKbBytes + k * 32);
              const uint64_t db = smem_desc_sw128(w1a + kb * 2 * kWPiece + k * 32);
              mma2_f16_ss(tmem_u, da, db, idesc_w, kk != 0);
            }
            mma2_commit(bar + kBarD1aFull);
            mma2_commit(bar + kBarD1bFull);
            mma2_commit(bar + kBarA1Empty + s);        // z consumed in both CTAs
          }
          __syncwarp();
          mbar_wait_c(bar + kBarA2aFull, ph);
          mbar_wait_c(bar + kBarD2Empty + g, ph2 ^ 1);
          tc_fence_after();
          if (issuer) {
#pragma unroll
            for (int kk = 0; kk < H / 16; ++kk) {
              const uint64_t db = smem_desc_sw128(w2a + (kk >> 2) * kWPiece + (kk & 3) * 32);
              mma2_f16_ts(tmem_u + kD2Col + g * kHidden, tmem_u + kk * 8, db, idesc, kk != 0);
            }
          }
          __syncwarp();
          mbar_wait_c(bar + kBarA2bFull, ph);
          tc_fence_after();
          if (issuer) {
#pragma unroll
            for (int kk = H / 16; kk < HID / 16; ++kk) {
              const uint64_t db = smem_desc_sw128(w2a + (kk >> 2) * kWPiece + (kk & 3) * 32);
              mma2_f16_ts(tmem_u + kD2Col + g * kHidden, tmem_u + kk * 8, db, idesc, 1u);
            }
            mma2_commit(bar + kBarD2Full + g);
          }
          __syncwarp();
        }
      }
    }
    __syncwarp();
  } else if (warp == kLoadWarp) {
    // ================= h tiles (TMA) =================================================
    reg_dec<40>();
    if (lane == 0) {
      prefetch_tmap(&maps.h);
      uint32_t it = 0;
      for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
        const uint32_t hb = it % kHBufs;
        const int row0 = (2 * pair + int(rank)) * kTileM;
        uint8_t *dst = hs + hb * kTileBytes;
        mbar_wait_parked(bar + kBarHEmpty + hb, ((it / kHBufs) & 1) ^ 1);
        mbar_arrive_expect_tx(bar + kBarHFull + hb, kTileBytes);
        tma_load_2d(dst, &maps.h, 0, row0, bar + kBarHFull + hb);
        tma_load_2d(dst + kKbBytes, &maps.h, 64, row0, bar + kBarHFull + hb);
      }
    }
    __syncwarp();
  } else if (warp == kStoreWarp) {
    // ================= output store (TMA) ============================================
    reg_dec<40>();
    if (lane == 0) {
      prefetch_tmap(&maps.out);
      uint32_t it = 0;
      for (int pair = cluster_id; pair < pairs; pair += clusters, ++it) {
        const uint32_t hb = it % kHBufs;
        const int row0 = (2 * pair + int(rank)) * kTileM;
        const uint8_t *src = hs + hb * kTileBytes;
        mbar_wait_parked(bar + kBarOReady + hb, (it / kHBufs) & 1);
        if (row0 < n) {
          tma_store_2d(&maps.out, 0, row0, src);
          tma_store_2d(&maps.out, 64, row0, src + kKbBytes);
        }
        bulk_commit();
        bulk_wait_read<0>();                      // shared memory has been read: the buffer is free
        mbar_arrive(bar + kBarHEmpty + hb);
      }
      bulk_wait_all();
    }
    __syncwarp();
  } else {
    reg_dec<40>();                                // spare warp of the utility warpgroup
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                             // the peer may still be arriving on our barriers
  if (warp == kMmaWarp) tmem_dealloc2(tmem, kTmemCols);
}

}  // namespace v6

int fused6_layer(const gfx_model *m, int layer, const __half *h, const int32_t *row_ptr,
                 const int32_t *col_src, const uint8_t *col_type, int64_t n, __half *h_out,
                 cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(h_out)) & 15)
    return fail(GFX_ERR_ARGUMENT, "fused layer: activation buffers must be 16-byte aligned");
  if (h == h_out) return fail(GFX_ERR_ARGUMENT, "fused layer: h and h_out must not alias");
  if (n > (int64_t(1) << v6::kSrcBits))
    return fail(GFX_ERR_UNSUPPORTED, "fused layer (CTA pairs): at most 2^27 nodes per call");
  if (m->edge_dim >= v6::kTabRows)
    return fail(GFX_ERR_UNSUPPORTED, "fused layer (CTA pairs): at most 10 edge types");
  v6::Maps maps;
  int rc = tma::make_rows128_map(&maps.h, h, n, v6::kTileM);
  if (!rc) rc = tma::make_rows128_map(&maps.out, h_out, n, v6::kTileM);
  if (rc) return rc;
  v6::Consts c;
  const gfx_host_vectors &hv = m->host;
  for (int i = 0; i < kMlpHidden; ++i) c.b1[i] = hv.b1[size_t(layer) * kMlpHidden + i];
  for (int i = 0; i < kHidden; ++i) {
    c.b2[i] = hv.b2[size_t(layer) * kHidden + i];
    c.g[i] = hv.ln_g[size_t(layer) * kHidden + i];
    c.be[i] = hv.ln_b[size_t(layer) * kHidden + i];
  }
  const size_t wi = size_t(layer) * kMlpHidden * kHidden;
  v6::Args a{};
  a.h = h; a.row_ptr = row_ptr; a.col_src = col_src; a.col_type = col_type;
  a.table16 = m->table16 + size_t(layer) * m->edge_dim * kHidden;
  a.w1_img = m->w1_img + wi; a.w2_img = m->w2_img + wi;
  a.n = n; a.edge_dim = m->edge_dim;
  const uint32_t e16 = __half_as_ushort(__float2half_rn(m->eps1[layer]));
  a.eps1_h2 = e16 | (e16 << 16);
  GFX_CUDA(cudaFuncSetAttribute(v6::fused_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                v6::Smem::total));
  const int64_t tiles = (n + v6::kTileM - 1) / v6::kTileM;
  const int64_t pairs = (tiles + 1) / 2;
  int cap = 0;
  rc = resident_pairs<v6::fused_pair_kernel>(v6::kWarps * 32, v6::Smem::total, &cap);
  if (rc) return rc;
  const int clusters = int(pairs < cap ? pairs : cap);
  v6::fused_pair_kernel<<<2 * clusters, v6::kWarps * 32, v6::Smem::total, st>>>(maps, c, a);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

}  // namespace gfx

extern "C" int gfx_layer_fused_pair(const gfx_model *m, int layer, const void *h,
                                    const int32_t *row_ptr, const int32_t *col_src,
                                    const uint8_t *col_type, int64_t n, void *h_out,
                                    void *stream) {
  using namespace gfx;
  if (!m || layer < 0 || layer >= m->layers)
    return fail(GFX_ERR_ARGUMENT, "gfx_layer_fused_pair: bad model or layer");
  if (n <= 0) return GFX_OK;
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_FUSED_LAYER, st, 1);
  return fused6_layer(m, layer, static_cast<const __half *>(h), row_ptr, col_src, col_type, n,
                      static_cast<__half *>(h_out), st);
}
