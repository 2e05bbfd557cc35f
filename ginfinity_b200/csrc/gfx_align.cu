// K8  batched Smith-Waterman alignment of per-nucleotide embeddings (affine gaps).
// No reference counterpart: the reference only ships scoring parameters for an
// external aligner (src/ginfinity/api.py:47-50).  The contract is in gfx.h.
//
// One persistent CTA per SM pulls pairs from a counter.  A pair is cut into
// stripes of 128 query rows; a stripe runs over the target in tiles of 128
// columns.  A (stripe, tile) is one work item:
//   warp 4     producer: TMA loads of the query stripe and the target tile (two
//              64-column swizzled K blocks each), eight tcgen05.mma kind::f16 of
//              K = 16 into one of four 128-column TMEM buffers, so up to four
//              items of S are ready ahead of the DP.
//   warps 0-3  DP: warp w owns rows 32w..32w+31 of the stripe (TMEM lanes of
//              its quarter), one row per lane.  It copies its 32 x 128 slab of S
//              from TMEM into shared memory (lane i reads S(i, j) at a column
//              that differs per lane, which registers cannot index) and runs an
//              anti-diagonal wavefront: at step k lane i computes column k - i,
//              taking H(i-1, j) and F(i-1, j) from lane i-1 by shuffle.  The
//              wavefront runs across the tiles of a stripe, so fill and drain
//              (31 steps) are paid once per stripe.  Lane 31's row goes to warp
//              w+1 through a 3-slot ring of 128-column chunks in shared memory;
//              warp 3's bottom row goes to warp 0 of the next stripe through a
//              per-CTA row in global memory (L2), one finished chunk at a time.  Warps follow each other one
//              tile apart, ordered by per-warp progress counters.
// Each DP warp reduces its rows' best cell per pair into `parts`; a second
// kernel picks the end cell of each pair by the tie rule.
//
// Traceback (gfx_align_trace) runs the same kernel with kTrace: each lane also records a
// 4-bit code per cell of its row (kCode* below), 32 columns to a uint4, stored every 32
// steps into the pair's pointer block (q_len rows x ceil(t_len/32) uint4, row-major).  In
// the last block of a row of t_len % 32 = r != 0 columns, column j sits at nibble
// 32 - r + (j & 31): the codes are shifted in from the top and the block is stored as it is.
// A walk kernel then follows the codes back from the end cell, one warp per pair.
//
// Arithmetic per cell, fp32 round-to-nearest in this order (gfx.h):
//   s = S - theta;  E = max(H_left - go, E_left - ge);  F = max(H_up - go, F_up - ge)
//   H = max(0, H_diag + s, E, F)
// Starts are packed as (i << 16) | j.
#include <limits.h>
#include <math.h>

#include "gfx_common.cuh"
#include "gfx_tma.cuh"
#include "gfx_umma.cuh"

namespace gfx {
namespace align {

using namespace ptx;

constexpr int kTile = 128;
constexpr int kMaxLen = 4096;                      // records.MAXIMUM_LENGTH_NT
constexpr int kBoxBytes = 128 * 128;               // [128 rows x 64 cols] fp16
constexpr int kDpWarps = 4, kProdWarp = 4, kThreads = 5 * 32;
constexpr int kBufs = 4;                           // TMEM accumulators of 128 columns
constexpr int kRingSlots = 3;                      // 128-column chunks between consecutive DP warps
// A lane's row of S: the two tiles in flight side by side, so column j is at (j & 255).  260
// floats per row: the float4 writes of 8 lanes and the reads of 32 lanes at 32 different
// columns (k - lane) fall in different banks.
constexpr int kSlabRow = 2 * kTile + 4;

struct Smem {
  static constexpr int off_stage = 0;                                   // A: 2 boxes, B: 2 boxes
  static constexpr int off_slab = off_stage + 4 * kBoxBytes;            // [warp][32][260] f32
  // ring w (w = 1..3) carries warp w-1's bottom row to warp w; ring 0 holds warp 0's top row
  // (from the previous stripe), ring 4 warp 3's bottom row on its way to global memory
  static constexpr int off_ring = off_slab + kDpWarps * 32 * kSlabRow * 4;  // [5][3][128] float4
  static constexpr int off_bar = off_ring + (kDpWarps + 1) * kRingSlots * kTile * 16;
  static constexpr int off_desc = off_bar + 16 * 8;                     // [kBufs] int4
  static constexpr int off_prog = off_desc + kBufs * 16;                // [kDpWarps] uint32
  static constexpr int off_tmem = off_prog + kDpWarps * 4;
  static constexpr int total = off_tmem + 16;
};
static_assert(Smem::total <= 232448, "exceeds the 227 KB shared-memory limit of sm_100");

enum Bar { kBarFull = 0, kBarEmpty = 4, kBarTma = 8, kBarSmem = 9, kNumBars = 10 };

struct alignas(64) Maps {
  CUtensorMap q, t;
};

struct Args {
  const int64_t *pairs;
  int64_t num_pairs, q_rows, t_rows;
  float theta, go, ge;
  float4 *parts;          // [P][4]: (best H, end, start, -) per DP warp
  unsigned long long *counter;
  float4 *rowbuf;         // [gridDim.x][row_cap]: (H, F, start H, start F) of warp 3's bottom row
  int row_cap;            // columns of rowbuf per CTA: the longest target of a multi-stripe pair
  // kTrace only
  uint8_t *codes;         // pointer blocks
  const int64_t *code_off;  // [P] byte offset of each pair's block in `codes`; -1: it did not fit
};

// Cell codes of the traceback: bits 0-1 where H came from, bit 2 E opened (else extended),
// bit 3 F opened.  H's source follows the tie rule: zero when H = 0, else the first of
// diagonal, E, F that attains it.
enum Code : uint32_t { kCodeZero = 0, kCodeDiag = 1, kCodeE = 2, kCodeF = 3, kCodeEOpen = 4, kCodeFOpen = 8 };

// Accuracy of S, relative: |S - q.t| <= kAlignRel |q| |t|.  The tensor-core sum is the same
// fp16-product, fp32-accumulate dot product as the top-k scan, so the argument of kCertRel in
// gfx_topk.cu carries over: within 2^-16 sum |q_k t_k| <= 2^-16 |q| |t| on the accumulator
// measured on earlier generations, with a 4x margin.  An alignment adds at most
// min(q_len, t_len) diagonal S terms, so its score is within min(q_len, t_len) kAlignRel
// max|q| max|t| of the same alignment in exact arithmetic; the DP adds (q_len + t_len) fp32
// roundings of 2^-24 relative.  This rests on that argument, not on a measurement.
[[maybe_unused]] constexpr float kAlignRel = 1.f / 16384.f;

// Workspace: the pair counter, then parts, then the per-CTA rows.  gfx_align_trace puts the
// pointer-block offsets after parts, then per-CTA rows of kMaxLen columns, then the blocks.
constexpr size_t kHeaderBytes = 256;
inline size_t parts_bytes(int64_t P) { return align256(size_t(P) * 4 * 16); }
inline int grid_for(int64_t P) { return int(P < kNumSMs ? (P > 0 ? P : 1) : kNumSMs); }
inline size_t trace_fixed_bytes(int64_t P) {
  return kHeaderBytes + parts_bytes(P) + align256(size_t(P) * 8) + size_t(grid_for(P)) * kMaxLen * 16;
}

// the limits of gfx.h, and a per-CTA row for a multi-stripe pair (the producer writes the same
// test out in full: as a call it changes the score instance's predicate allocation)
__device__ __forceinline__ bool pair_valid(int64_t qs, int64_t ql, int64_t ts, int64_t tl, const Args &a) {
  return qs >= 0 && ql >= 0 && ql <= kMaxLen && qs <= a.q_rows - ql && ts >= 0 && tl >= 0 &&
         tl <= kMaxLen && ts <= a.t_rows - tl && (ql <= kTile || tl <= a.row_cap);
}
__device__ __forceinline__ int64_t code_bytes(int64_t ql, int64_t tl) { return ql * ((tl + 31) / 32) * 16; }

__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ uint32_t ld_vol(const uint32_t *p) { return *reinterpret_cast<const volatile uint32_t *>(p); }
__device__ __forceinline__ void st_vol(uint32_t *p, uint32_t v) { *reinterpret_cast<volatile uint32_t *>(p) = v; }
__device__ __forceinline__ void wait_at_least(const uint32_t *p, uint32_t v) {
  while (ld_vol(p) < v) {
  }
  __threadfence_block();
}

// lane 31's writes so far are visible to the warp that waits for `v`
__device__ __forceinline__ void publish(uint32_t *p, uint32_t v, int lane) {
  __threadfence_block();
  __syncwarp();
  if (lane == 0) st_vol(p, v);
}

// DP state of one lane (one row of the stripe)
struct Dp {
  float H, E, F, Hd;               // H, E, F of the last cell; H of the cell above-left of the next
  uint32_t sH, sE, sF, sHd;        // their starts, (i << 16) | j
  float cur;                       // best H of the row so far (+inf: row outside the segment)
  uint32_t best_end, best_start, ibase;
  uint32_t c0, c1, c2, c3;         // kTrace: codes of the last 32 cells, the newest in c3's top nibble
  uint4 *crow;                     // kTrace: this row's codes
  int clast;                       // kTrace: last column stored (t_len - 1; -1 past the segment)
};

// Anti-diagonal steps k0 .. k1-1: lane computes cell (row, k - lane).  FILL: some lanes are
// left of column 0 (k < 31); DRAIN: some are right of the last column (k >= t_len).
template <bool TRACE, bool FILL, bool DRAIN>
__device__ __forceinline__ void dp_steps(Dp &d, int k0, int k1, int lane, const float *srow,
                                         const float4 *top, float4 *out, int t_len, float theta,
                                         float go, float ge) {
  for (int k = k0; k < k1; ++k) {
    const int j = k - lane;
    float upH = __shfl_up_sync(0xffffffffu, d.H, 1);
    float upF = __shfl_up_sync(0xffffffffu, d.F, 1);
    uint32_t upsH = __shfl_up_sync(0xffffffffu, d.sH, 1);
    uint32_t upsF = __shfl_up_sync(0xffffffffu, d.sF, 1);
    if (lane == 0) {
      const float4 v = top[k & (kTile - 1)];
      upH = v.x;
      upF = v.y;
      upsH = __float_as_uint(v.z);
      upsF = __float_as_uint(v.w);
    }
    float sc = srow[j & (2 * kTile - 1)] - theta;
    // left of column 0 the cells must stay H = 0: a score of -inf gives H = 0 and E, F = -go
    // there, which enter column 0 exactly as E(i,-1) = -inf would
    if (FILL) sc = j >= 0 ? sc : -INFINITY;
    const float eo = d.H - go, ee = d.E - ge;
    const float En = fmaxf(eo, ee);
    const uint32_t sEn = eo >= ee ? d.sH : d.sE;
    const float fo = upH - go, fe = upF - ge;
    const float Fn = fmaxf(fo, fe);
    const uint32_t sFn = fo >= fe ? upsH : upsF;
    const float dg = d.Hd + sc;
    const float Hn = fmaxf(max3(dg, En, Fn), 0.f);
    const uint32_t sdiag = d.Hd == 0.f ? d.ibase | uint32_t(j) : d.sHd;
    const uint32_t sgap = En == Hn ? sEn : sFn;
    const uint32_t sHn = dg == Hn ? sdiag : sgap;
    d.Hd = upH;
    d.sHd = upsH;
    d.H = Hn;
    d.E = En;
    d.F = Fn;
    d.sH = sHn;
    d.sE = sEn;
    d.sF = sFn;
    if constexpr (TRACE) {
      const uint32_t src = Hn == 0.f ? kCodeZero : dg == Hn ? kCodeDiag : En == Hn ? kCodeE : kCodeF;
      const uint32_t c = src | (eo >= ee ? kCodeEOpen : 0u) | (fo >= fe ? kCodeFOpen : 0u);
      d.c0 = __funnelshift_r(d.c0, d.c1, 4);
      d.c1 = __funnelshift_r(d.c1, d.c2, 4);
      d.c2 = __funnelshift_r(d.c2, d.c3, 4);
      d.c3 = __funnelshift_r(d.c3, c, 4);
      // the last column of a 32-column block, or of the row
      if (j == min(j | 31, d.clast) && (!FILL || j >= 0)) d.crow[j >> 5] = make_uint4(d.c0, d.c1, d.c2, d.c3);
    }
    if (Hn > d.cur && (!DRAIN || unsigned(j) < unsigned(t_len))) {
      d.cur = Hn;
      d.best_end = d.ibase | uint32_t(j);
      d.best_start = sHn;
    }
    if (lane == 31) out[(k - 31) & (kTile - 1)] = make_float4(Hn, Fn, __uint_as_float(sHn), __uint_as_float(sFn));
  }
}

template <bool kTrace>
__global__ void __launch_bounds__(kThreads, 1)
align_kernel(const __grid_constant__ Maps maps, const Args a) {
  using L = Smem;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::off_bar);
  int *desc = reinterpret_cast<int *>(smem + L::off_desc);
  uint32_t *prog = reinterpret_cast<uint32_t *>(smem + L::off_prog);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::off_tmem);
  float4 *ring = reinterpret_cast<float4 *>(smem + L::off_ring);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == kProdWarp) {
    tmem_alloc(tmem_slot, kBufs * kTile);
  } else if (tid == 0) {
    for (int r = 0; r < kBufs; ++r) {
      mbar_init(bar + kBarFull + r, 2);            // MMA commit + producer's descriptor
      mbar_init(bar + kBarEmpty + r, kDpWarps);
    }
    mbar_init(bar + kBarTma, 1);
    mbar_init(bar + kBarSmem, 1);
    for (int w = 0; w < kDpWarps; ++w) prog[w] = 0;
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == kProdWarp) {
    // ============================ producer: TMA + MMA ==============================
    // (whole warp in the loop, one elected lane issues: warp-uniform operands stay in
    // uniform registers, see the top-k scan)
    uint32_t elected;
    asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(elected));
    const bool issuer = elected != 0u;
    if (issuer) {
      prefetch_tmap(&maps.q);
      prefetch_tmap(&maps.t);
    }
    constexpr uint32_t idesc = idesc_f16(128, kTile);
    const uint32_t sa = smem_u32(smem + L::off_stage);
    uint32_t n = 0;
    for (;;) {
      unsigned long long p = 0;
      if (lane == 0) p = atomicAdd(a.counter, 1ull);
      p = __shfl_sync(0xffffffffu, p, 0);
      if (p >= (unsigned long long)a.num_pairs) break;
      int64_t v = lane < 4 ? a.pairs[p * 4 + lane] : 0;
      const int64_t qs = __shfl_sync(0xffffffffu, v, 0), ql = __shfl_sync(0xffffffffu, v, 1);
      const int64_t ts = __shfl_sync(0xffffffffu, v, 2), tl = __shfl_sync(0xffffffffu, v, 3);
      const bool valid = qs >= 0 && ql >= 0 && ql <= kMaxLen && qs <= a.q_rows - ql && ts >= 0 && tl >= 0 &&
                         tl <= kMaxLen && ts <= a.t_rows - tl && (ql <= kTile || tl <= a.row_cap) &&
                         (!kTrace || a.code_off[p] >= 0);
      if (!valid || ql == 0 || tl == 0) {
        // nothing to align: score 0 (or NaN for a pair the caller should not have passed)
        if (lane < kDpWarps)
          a.parts[p * 4 + lane] = make_float4(valid ? 0.f : __int_as_float(0x7fc00000), __uint_as_float(~0u), 0.f, 0.f);
        continue;
      }
      const int stripes = int((ql + kTile - 1) / kTile), tiles = int((tl + kTile - 1) / kTile);
      for (int s = 0; s < stripes; ++s) {
        for (int t = 0; t < tiles; ++t, ++n) {
          const uint32_t r = n & (kBufs - 1);
          mbar_wait_parked(bar + kBarEmpty + r, ((n / kBufs) & 1) ^ 1);
          if (lane == 0) {
            desc[r * 4 + 0] = int(p);
            desc[r * 4 + 1] = int(ql);
            desc[r * 4 + 2] = int(tl);
          }
          mbar_wait_parked(bar + kBarSmem, (n & 1) ^ 1);   // the previous item's MMAs are done
          if (issuer) {
            uint8_t *st = smem + L::off_stage;
            mbar_arrive_expect_tx(bar + kBarTma, 4 * kBoxBytes);
            tma_load_2d(st, &maps.q, 0, int(qs + s * kTile), bar + kBarTma);
            tma_load_2d(st + kBoxBytes, &maps.q, 64, int(qs + s * kTile), bar + kBarTma);
            tma_load_2d(st + 2 * kBoxBytes, &maps.t, 0, int(ts + t * kTile), bar + kBarTma);
            tma_load_2d(st + 3 * kBoxBytes, &maps.t, 64, int(ts + t * kTile), bar + kBarTma);
          }
          __syncwarp();
          mbar_wait(bar + kBarTma, n & 1);
          tc_fence_after();
          if (issuer) {
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              const int kb = kk >> 2, k = kk & 3;
              const uint64_t da = smem_desc_sw128(sa + kb * kBoxBytes + k * 32);
              const uint64_t db = smem_desc_sw128(sa + (2 + kb) * kBoxBytes + k * 32);
              mma_f16_ss(tmem + r * kTile, da, db, idesc, kk != 0);
            }
            mma_commit(bar + kBarSmem);
            mma_commit(bar + kBarFull + r);
          }
          if (lane == 0) mbar_arrive(bar + kBarFull + r);   // releases the descriptor
          __syncwarp();
        }
      }
    }
    const uint32_t r = n & (kBufs - 1);                  // end of work
    mbar_wait_parked(bar + kBarEmpty + r, ((n / kBufs) & 1) ^ 1);
    if (lane == 0) {
      desc[r * 4] = -1;
      mbar_arrive(bar + kBarFull + r);
      mbar_arrive(bar + kBarFull + r);
    }
    __syncwarp();
  } else {
    // ================================== DP warps ===================================
    const int w = warp;
    float *slab = reinterpret_cast<float *>(smem + L::off_slab) + w * 32 * kSlabRow;
    float4 *in_ring = ring + w * kRingSlots * kTile;
    float4 *next_ring = ring + (w + 1) * kRingSlots * kTile;
    float4 *rowbuf = a.rowbuf + size_t(blockIdx.x) * a.row_cap;
    const uint32_t tlane = tmem + (uint32_t(32 * w) << 16);
    const float theta = a.theta, go = a.go, ge = a.ge, ninf = -INFINITY;
    uint32_t n = 0;
    for (;;) {
      mbar_wait(bar + kBarFull + (n & (kBufs - 1)), (n / kBufs) & 1);
      const int *dsc = desc + (n & (kBufs - 1)) * 4;
      const int p = reinterpret_cast<const volatile int *>(dsc)[0];
      if (p < 0) break;
      const int q_len = reinterpret_cast<const volatile int *>(dsc)[1];
      const int t_len = reinterpret_cast<const volatile int *>(dsc)[2];
      const int stripes = (q_len + kTile - 1) / kTile, tiles = (t_len + kTile - 1) / kTile;
      uint4 *cblock = nullptr;
      if constexpr (kTrace) cblock = reinterpret_cast<uint4 *>(a.codes + a.code_off[p]);
      float best = 0.f;                       // best H of this lane's rows, strictly positive to count
      uint32_t best_end = ~0u, best_start = 0;
      for (int s = 0; s < stripes; ++s) {
        const uint32_t n0 = n;                // item of tile 0 of this stripe
        if (s * kTile + w * 32 >= q_len) {
          // no row of this warp is in the pair: only keep the pipeline moving
          for (int t = 0; t < tiles; ++t, ++n) {
            mbar_wait(bar + kBarFull + (n & (kBufs - 1)), (n / kBufs) & 1);
            __syncwarp();
            if (lane == 0) {
              mbar_arrive(bar + kBarEmpty + (n & (kBufs - 1)));
              st_vol(prog + w, n + 1);
            }
          }
          __syncwarp();
          continue;
        }
        const int row = s * kTile + w * 32 + lane;
        Dp st;
        st.ibase = uint32_t(row) << 16;
        st.cur = row < q_len ? best : INFINITY;     // rows past the segment never score
        st.best_end = best_end;
        st.best_start = best_start;
        st.H = 0.f;
        st.E = st.F = ninf;
        st.Hd = 0.f;
        st.sH = st.sE = st.sF = st.sHd = 0;
        if constexpr (kTrace) {
          st.c0 = st.c1 = st.c2 = st.c3 = 0;
          st.crow = cblock + size_t(row) * ((t_len + 31) / 32);
          st.clast = row < q_len ? t_len - 1 : -1;
        }
        const float *srow = slab + lane * kSlabRow;
        const float4 *in_cur = in_ring;
        float4 *out_even = nullptr, *out_odd = nullptr;   // lane 31's destination for even / odd tiles
        float4 *out = nullptr;
        // warp 3: tile u's bottom row, complete, to the global row for the next stripe
        auto to_rowbuf = [&](int u) {
          if (w + 1 == kDpWarps && s + 1 < stripes) {
            __syncwarp();
            const float4 *src = u & 1 ? out_odd : out_even;
#pragma unroll
            for (int c = lane; c < kTile; c += 32) __stcg(rowbuf + u * kTile + c, src[c]);
          }
        };
        const int kend = t_len + 31;
        // Steps run in segments between events: lane 0 enters a tile (k = 128 t), lane 31
        // enters a tile (k = 128 t + 31: the previous tile's bottom row is complete), the
        // drain starts (k = t_len).  The fill (k < 31) and the drain are step variants.
        for (int k = 0; k < kend;) {
          if ((k & (kTile - 1)) == 0 && k < t_len) {
            // ---- lane 0 enters tile t = item n ----
            const int t = k / kTile;
            const uint32_t r = n & (kBufs - 1);
            mbar_wait(bar + kBarFull + r, (n / kBufs) & 1);
            tc_fence_after();
            float *dst = slab + lane * kSlabRow + (t & 1) * kTile;
#pragma unroll 1
            for (int cb = 0; cb < 4; ++cb) {
              float v[32];
              tmem_ld32(tlane + r * kTile + cb * 32, v);
              tmem_ld_wait();
#pragma unroll
              for (int c = 0; c < 32; c += 4)
                *reinterpret_cast<float4 *>(dst + cb * 32 + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + kBarEmpty + r);
            const uint32_t slot = n % kRingSlots;
            float4 *in_slot = in_ring + slot * kTile;
            if (w > 0) {
              wait_at_least(prog + w - 1, n + 1);      // warp w-1 has finished this tile
            } else if (s > 0) {
              wait_at_least(prog + kDpWarps - 1, n + 1 - tiles);   // warp 3, same tile, previous stripe
#pragma unroll
              for (int c = lane; c < kTile; c += 32) in_slot[c] = __ldcg(rowbuf + t * kTile + c);
            } else {
#pragma unroll
              for (int c = lane; c < kTile; c += 32) in_slot[c] = make_float4(0.f, ninf, 0.f, 0.f);
            }
            if (w + 1 < kDpWarps)
              wait_at_least(prog + w + 1, n + 1 > kRingSlots ? n + 1 - kRingSlots : 0);   // slot is free
            float4 *o = next_ring + slot * kTile;
            if (t & 1) out_odd = o; else out_even = o;
            if (t == 0) out = o;         // lane 31's fill steps write columns it rewrites later
            in_cur = in_slot;
            __syncwarp();
            ++n;
          }
          if (k >= 31 && ((k - 31) & (kTile - 1)) == 0) {
            // ---- lane 31 enters tile u: tile u-1's bottom row is complete ----
            const int u = (k - 31) / kTile;
            if (u > 0) {
              to_rowbuf(u - 1);
              publish(prog + w, n0 + uint32_t(u), lane);
            }
            out = u & 1 ? out_odd : out_even;
          }
          int next = k < 31 ? 31 : k + kTile - ((k - 31) & (kTile - 1));
          const int tile_next = (k / kTile + 1) * kTile;
          if (tile_next < t_len && tile_next < next) next = tile_next;
          if (k < t_len && t_len < next) next = t_len;
          if (kend < next) next = kend;
          if (k < 31) {
            if (k < t_len) dp_steps<kTrace, true, false>(st, k, next, lane, srow, in_cur, out, t_len, theta, go, ge);
            else dp_steps<kTrace, true, true>(st, k, next, lane, srow, in_cur, out, t_len, theta, go, ge);
          } else {
            if (k < t_len) dp_steps<kTrace, false, false>(st, k, next, lane, srow, in_cur, out, t_len, theta, go, ge);
            else dp_steps<kTrace, false, true>(st, k, next, lane, srow, in_cur, out, t_len, theta, go, ge);
          }
          k = next;
        }
        to_rowbuf(tiles - 1);
        publish(prog + w, n0 + uint32_t(tiles), lane);
        best_end = st.best_end;
        best_start = st.best_start;
        const float cur = st.cur;
        if (row < q_len) best = cur;
      }
      // the warp's best cell: largest H, then smallest (i, j)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float oh = __shfl_xor_sync(0xffffffffu, best, o);
        const uint32_t oe = __shfl_xor_sync(0xffffffffu, best_end, o);
        const uint32_t os = __shfl_xor_sync(0xffffffffu, best_start, o);
        if (oh > best || (oh == best && oe < best_end)) {
          best = oh;
          best_end = oe;
          best_start = os;
        }
      }
      if (lane == 0)
        a.parts[size_t(p) * 4 + w] = make_float4(best, __uint_as_float(best_end), __uint_as_float(best_start), 0.f);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kProdWarp) tmem_dealloc(tmem, kBufs * kTile);
}

// One thread per pair: the end cell over the four DP warps (largest H, then smallest
// (i, j)), and the half-open coordinates of the alignment that reaches it.
__global__ void __launch_bounds__(256)
align_finish_kernel(const float4 *__restrict__ parts, int64_t P, float *__restrict__ score,
                    int4 *__restrict__ coords) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float4 b = parts[p * 4];
  for (int w = 1; w < kDpWarps; ++w) {
    const float4 o = parts[p * 4 + w];
    if (o.x > b.x || (o.x == b.x && __float_as_uint(o.y) < __float_as_uint(b.y))) b = o;
  }
  if (b.x > 0.f) {
    const uint32_t e = __float_as_uint(b.y), st = __float_as_uint(b.z);
    score[p] = b.x;
    coords[p] = make_int4(int(st >> 16), int(e >> 16) + 1, int(st & 0xffffu), int(e & 0xffffu) + 1);
  } else {
    score[p] = b.x == 0.f ? 0.f : b.x;     // NaN marks a pair outside the tables
    coords[p] = make_int4(-1, -1, -1, -1);
  }
}

// kTrace: byte offset of each pair's pointer block, in pair order (one block of 1024 threads,
// an exclusive scan 1024 pairs at a time).  A block that ends past `capacity` gets -1.
__global__ void __launch_bounds__(1024) align_code_offsets_kernel(const Args a, int64_t capacity) {
  __shared__ int64_t warp_sum[32];
  __shared__ int64_t carry;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int64_t *off = const_cast<int64_t *>(a.code_off);
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < a.num_pairs; base += 1024) {
    const int64_t p = base + tid;
    int64_t bytes = 0;
    if (p < a.num_pairs) {
      const int64_t qs = a.pairs[p * 4], ql = a.pairs[p * 4 + 1], ts = a.pairs[p * 4 + 2], tl = a.pairs[p * 4 + 3];
      if (pair_valid(qs, ql, ts, tl, a)) bytes = code_bytes(ql, tl);
    }
    int64_t x = bytes;                     // inclusive scan over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int64_t v = warp_sum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += y;
      }
      warp_sum[lane] = v;
    }
    __syncthreads();
    const int64_t end = carry + (warp > 0 ? warp_sum[warp - 1] : 0) + x;
    if (p < a.num_pairs) off[p] = end <= capacity ? end - bytes : -1;
    __syncthreads();
    if (tid == 1023) carry = end;
    __syncthreads();
  }
}

// The traceback: one warp per pair, from the end cell the finish kernel picked.  The lanes
// stage the 32 rows x 32 columns of codes that end at the current cell (one uint4 each);
// lane 0 walks them until the path leaves that block, collecting ops in reverse.  A walk
// that does not end at the reported start (or leaves the segments) gets length -1.
constexpr int kWalkWarps = 4;
constexpr int kMaxPath = 2 * kMaxLen - 1;

__global__ void __launch_bounds__(kWalkWarps * 32)
align_walk_kernel(const int64_t *__restrict__ pairs, int64_t P, const int64_t *__restrict__ code_off,
                  const uint8_t *__restrict__ codes, const float *__restrict__ score,
                  const int4 *__restrict__ coords, const int64_t *__restrict__ op_off,
                  uint8_t *__restrict__ ops, int32_t *__restrict__ out_len) {
  __shared__ uint4 stage_all[kWalkWarps][32];
  __shared__ uint8_t rev_all[kWalkWarps][kMaxPath + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t p = int64_t(blockIdx.x) * kWalkWarps + warp;
  if (p >= P) return;
  if (!(score[p] > 0.f)) {
    if (lane == 0) out_len[p] = 0;
    return;
  }
  const int4 c = coords[p];
  const int t_len = int(pairs[p * 4 + 3]);
  const int stride = (t_len + 31) / 32, rem = t_len & 31;
  const uint4 *blk = reinterpret_cast<const uint4 *>(codes + code_off[p]);
  uint4 *stage = stage_all[warp];
  uint8_t *rev = rev_all[warp];
  int i = c.y - 1, j = c.w - 1, state = kCodeDiag, n = 0, status = 0;   // status: 1 done, 2 failed
  for (;;) {
    i = __shfl_sync(0xffffffffu, i, 0);
    j = __shfl_sync(0xffffffffu, j, 0);
    status = __shfl_sync(0xffffffffu, status, 0);
    if (status) break;
    const int r = i - 31 + lane;
    stage[lane] = r >= 0 ? blk[size_t(r) * stride + (j >> 5)] : make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();
    if (lane == 0) {
      const int i0 = i - 31, cb = j >> 5;
      const int shift = rem != 0 && cb == stride - 1 ? 32 - rem : 0;
      const uint32_t *words = reinterpret_cast<const uint32_t *>(stage);
      for (;;) {
        if (i < 0 || j < 0) {
          // only a diagonal step may leave the segments, and only from the reported start
          status = state == kCodeDiag && n > 0 && rev[n - 1] == 0 && i + 1 == c.x && j + 1 == c.z ? 1 : 2;
          break;
        }
        if (i < i0 || (j >> 5) != cb) break;
        if (n == kMaxPath) {
          status = 2;
          break;
        }
        const int nib = (j & 31) + shift;
        const uint32_t code = (words[(i - i0) * 4 + (nib >> 3)] >> ((nib & 7) * 4)) & 15u;
        if (state == kCodeDiag) {
          const uint32_t src = code & 3u;
          if (src == kCodeZero) {
            // H = 0 here: the diagonal step into the previous cell started the alignment
            status = n > 0 && rev[n - 1] == 0 && i + 1 == c.x && j + 1 == c.z ? 1 : 2;
            break;
          }
          if (src == kCodeDiag) {
            rev[n++] = 0;
            --i;
            --j;
          } else {
            state = int(src);
          }
        } else if (state == kCodeE) {
          rev[n++] = 2;
          state = code & kCodeEOpen ? kCodeDiag : kCodeE;
          --j;
        } else {
          rev[n++] = 1;
          state = code & kCodeFOpen ? kCodeDiag : kCodeF;
          --i;
        }
      }
    }
    __syncwarp();
  }
  n = __shfl_sync(0xffffffffu, n, 0);
  uint8_t *dst = ops + op_off[p];
  if (status == 1)
    for (int k = lane; k < n; k += 32) dst[k] = rev[n - 1 - k];
  if (lane == 0) out_len[p] = status == 1 ? n : -1;
}

}  // namespace align
}  // namespace gfx

using namespace gfx;

extern "C" size_t gfx_align_workspace_bytes(int64_t num_pairs, int64_t max_t_len) {
  if (num_pairs < 0) num_pairs = 0;
  if (max_t_len < 0) max_t_len = 0;
  if (max_t_len > align::kMaxLen) max_t_len = align::kMaxLen;
  const size_t cols = size_t((max_t_len + align::kTile - 1) / align::kTile) * align::kTile;
  return align::kHeaderBytes + align::parts_bytes(num_pairs) + size_t(align::grid_for(num_pairs)) * cols * 16;
}

extern "C" size_t gfx_align_trace_workspace_bytes(int64_t num_pairs, int64_t code_bytes) {
  if (num_pairs < 0) num_pairs = 0;
  if (code_bytes < 0) code_bytes = 0;
  return align::trace_fixed_bytes(num_pairs) + size_t(code_bytes);
}

namespace {

// gfx_align and gfx_align_trace: the same checks and launches; `trace` adds the pointer
// blocks, the code pass and the walk.
struct TraceOut {
  uint8_t *ops;
  const int64_t *op_offsets;
  int32_t *len;
};

int run_align(const char *name, const void *queries, int64_t q_rows, const void *targets, int64_t t_rows,
              const int64_t *pairs, int64_t num_pairs, float offset, float gap_open, float gap_extend,
              float *out_score, int32_t *out_coords, const TraceOut *trace, void *workspace,
              size_t workspace_bytes, void *stream) {
  const std::string fn(name);
  if (num_pairs < 0 || q_rows < 0 || t_rows < 0 || q_rows > int64_t(INT_MAX) - 256 ||
      t_rows > int64_t(INT_MAX) - 256)
    return fail(GFX_ERR_ARGUMENT, fn + ": bad sizes (table rows must fit int32)");
  if (!std::isfinite(offset) || !std::isfinite(gap_open) || !std::isfinite(gap_extend))
    return fail(GFX_ERR_ARGUMENT, fn + ": offset, gap_open and gap_extend must be finite");
  if (!(gap_open > 0.f) || !(gap_extend > 0.f))
    return fail(GFX_ERR_ARGUMENT, fn + ": gap_open and gap_extend must be positive");
  if (num_pairs == 0) return GFX_OK;
  if (!pairs || !out_score || !out_coords || !workspace || (q_rows > 0 && !queries) || (t_rows > 0 && !targets) ||
      (trace && (!trace->ops || !trace->op_offsets || !trace->len)))
    return fail(GFX_ERR_ARGUMENT, fn + ": null pointer");
  if ((reinterpret_cast<uintptr_t>(queries) | reinterpret_cast<uintptr_t>(targets) |
       reinterpret_cast<uintptr_t>(out_coords) | reinterpret_cast<uintptr_t>(workspace)) & 15)
    return fail(GFX_ERR_ARGUMENT, fn + ": tables, out_coords and workspace must be 16-byte aligned");
  const int grid = align::grid_for(num_pairs);
  const size_t fixed = trace ? align::trace_fixed_bytes(num_pairs)
                             : align::kHeaderBytes + align::parts_bytes(num_pairs);
  if (workspace_bytes < fixed) return fail(GFX_ERR_WORKSPACE, fn + ": workspace too small");
  int64_t row_cap = int64_t((workspace_bytes - fixed) / (size_t(grid) * 16));
  row_cap = row_cap > align::kMaxLen ? align::kMaxLen : row_cap / align::kTile * align::kTile;
  cudaStream_t st = as_stream(stream);
  char *ws = static_cast<char *>(workspace);
  align::Args a{};
  a.pairs = pairs;
  a.num_pairs = num_pairs;
  a.q_rows = q_rows;
  a.t_rows = t_rows;
  a.theta = offset;
  a.go = gap_open;
  a.ge = gap_extend;
  a.counter = reinterpret_cast<unsigned long long *>(ws);
  a.parts = reinterpret_cast<float4 *>(ws + align::kHeaderBytes);
  a.rowbuf = reinterpret_cast<float4 *>(ws + fixed);
  a.row_cap = int(row_cap);
  if (trace) {
    // offsets, then per-CTA rows of kMaxLen columns, then the pointer blocks
    const size_t off_at = align::kHeaderBytes + align::parts_bytes(num_pairs);
    a.code_off = reinterpret_cast<const int64_t *>(ws + off_at);
    a.rowbuf = reinterpret_cast<float4 *>(ws + off_at + align256(size_t(num_pairs) * 8));
    a.row_cap = align::kMaxLen;
    a.codes = reinterpret_cast<uint8_t *>(ws + fixed);
  }
  // An empty table is described as one row of the workspace; no pair can read it
  // (a segment inside it has length 0).
  align::Maps maps;
  int rc = tma::make_rows128_map(&maps.q, q_rows ? queries : workspace, q_rows ? q_rows : 1, 128);
  if (!rc) rc = tma::make_rows128_map(&maps.t, t_rows ? targets : workspace, t_rows ? t_rows : 1, 128);
  if (rc) return rc;
  StageScope scope(GFX_STAGE_ALIGN, st, trace ? 4 : 2);
  GFX_CUDA(cudaMemsetAsync(ws, 0, align::kHeaderBytes, st));
  if (trace) {
    align::align_code_offsets_kernel<<<1, 1024, 0, st>>>(a, int64_t(workspace_bytes - fixed));
    GFX_LAUNCH_CHECK();
    GFX_CUDA(cudaFuncSetAttribute(align::align_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  align::Smem::total));
    align::align_kernel<true><<<grid, align::kThreads, align::Smem::total, st>>>(maps, a);
  } else {
    GFX_CUDA(cudaFuncSetAttribute(align::align_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  align::Smem::total));
    align::align_kernel<false><<<grid, align::kThreads, align::Smem::total, st>>>(maps, a);
  }
  GFX_LAUNCH_CHECK();
  align::align_finish_kernel<<<int((num_pairs + 255) / 256), 256, 0, st>>>(
      a.parts, num_pairs, out_score, reinterpret_cast<int4 *>(out_coords));
  GFX_LAUNCH_CHECK();
  if (trace) {
    align::align_walk_kernel<<<int((num_pairs + align::kWalkWarps - 1) / align::kWalkWarps),
                               align::kWalkWarps * 32, 0, st>>>(
        pairs, num_pairs, a.code_off, a.codes, out_score, reinterpret_cast<const int4 *>(out_coords),
        trace->op_offsets, trace->ops, trace->len);
    GFX_LAUNCH_CHECK();
  }
  return GFX_OK;
}

}  // namespace

extern "C" int gfx_align(const void *queries, int64_t q_rows, const void *targets, int64_t t_rows,
                         const int64_t *pairs, int64_t num_pairs, float offset, float gap_open,
                         float gap_extend, float *out_score, int32_t *out_coords, void *workspace,
                         size_t workspace_bytes, void *stream) {
  return run_align("gfx_align", queries, q_rows, targets, t_rows, pairs, num_pairs, offset, gap_open,
                   gap_extend, out_score, out_coords, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int gfx_align_trace(const void *queries, int64_t q_rows, const void *targets, int64_t t_rows,
                               const int64_t *pairs, int64_t num_pairs, float offset, float gap_open,
                               float gap_extend, float *out_score, int32_t *out_coords, uint8_t *out_ops,
                               const int64_t *op_offsets, int32_t *out_len, void *workspace,
                               size_t workspace_bytes, void *stream) {
  const TraceOut trace{out_ops, op_offsets, out_len};
  return run_align("gfx_align_trace", queries, q_rows, targets, t_rows, pairs, num_pairs, offset, gap_open,
                   gap_extend, out_score, out_coords, &trace, workspace, workspace_bytes, stream);
}
