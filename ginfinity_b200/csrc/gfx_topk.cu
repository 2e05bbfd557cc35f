// K5  similarity search: per-query top-k of a [Q,128] query set against a
// [D,128] embedding database of fp16 rows (gfx_topk) or fp32 rows (gfx_topk_f32)
// (cosine = dot product of unit vectors, or negative squared L2 distance).  No
// reference counterpart (north-star item 4).
//
//   scan    tcgen05 GEMM  S = Q_tile x DB_tile(128)^T  with the running top-k
//           fused into the TMEM epilogue: the score matrix never exists in
//           memory.  One persistent CTA per SM; a work item is (query tile,
//           database segment).  Warps: epilogue (one query per thread), then the
//           MMA issuer and the TMA loader.  Database tiles stream through a TMA
//           ring (the same tile is read by every resident CTA at about the same
//           time, so all but the first read hit L2); the queries of the item
//           stay in shared memory; accumulators are double-buffered in TMEM.
//           Two configurations of the same code:
//             F16Scan    fp16 rows (topk_scan_kernel): 256-query tiles, 8 epilogue warps, 3 stages,
//                        TMEM 2 x 2 x 128 columns, one MMA per K step.
//             SplitScan  fp32 rows (split_search_kernel): the operands are split-fp16 images,
//                        x = hi + lo, hi = fp16(x), lo = fp16(x - hi) (the split
//                        of gfx_split9.cu), [rows, 256] = hi | lo; per K step
//                        three kind::f16 MMAs, hi.hi + hi.lo + lo.hi, into one
//                        fp32 accumulator.  The database image is built once per
//                        index (gfx_topk_f32_prepare), the queries' per call in
//                        the workspace.  Hi and lo need twice the shared memory,
//                        so a work item holds 128 queries: queries 64 KB |
//                        2 stages x 64 KB | |d|^2 slots 4 KB | lists <= 28 KB =
//                        224 KB; 4 epilogue warps; TMEM 2 x 128 columns.
//   finish  exact re-scoring of the surviving candidates from the rows as given
//           (sequential fp32 FMA in dimension order: reproducible and restatable
//           on the CPU), selection of the k best by (score desc, index asc), and
//           a certificate per query (below).
//   fallback  for the queries whose certificate fails: an exact scan of the
//           whole database (the same FMA chain for every row) and the same
//           selection.  Launched unconditionally; its grid reads the number
//           of flagged queries on the device.
//   merge   k-way merge of per-rank lists after the all-gather.
//
// Tensor-core scores only choose the candidates (kc = k + >=4 spares per
// segment); the returned scores and order come from the exact pass.  The scan
// drops a row only when its tensor-core score is <= max(seed', last entry of a
// full list), so the largest such bound B over the segments bounds every
// dropped row.  A query is certified when B + eps < S_k, its k-th exact score
// in the scan's frame (+|q|^2 for L2): no dropped row can then reach the top k.
// Otherwise (near-ties the tensor cores cannot order, e.g. many near-duplicate
// rows, or a row of very large norm inflating eps) the query is rescored
// exactly against every row.  The result is exact for every input.
#include <limits.h>
#include <math.h>

#include <string>
#include <type_traits>

#include "gfx_common.cuh"
#include "gfx_tma.cuh"
#include "gfx_umma.cuh"

namespace gfx {
namespace topk {

using namespace ptx;

constexpr int kDbTile = 128;
constexpr int kBoxBytes = 128 * 128;              // [128 rows x 64 cols] fp16: one TMA box
constexpr int kD2Slots = 8;                       // loader runs <= 5 tiles ahead of the epilogue
constexpr int kMaxCand = 28, kMaxK = 24;
constexpr int kWaves = 8;                         // work items per CTA aimed for
constexpr int kSampleTiles = 128;                 // database tiles of the threshold-seeding pre-pass

// Compile-time shape of a scan over rows of type ROW.  The MMA operands are fp16
// images of kParts x 64-column K blocks per row: the rows themselves (fp16), or
// hi | lo (fp32, kParts = 2).  Box (row block rb, part p, K block kb) holds
// image columns [(p * 2 + kb) * 64, +64) of rows [qt * kQTile + rb * 128, +128)
// and sits in shared memory at box index (rb * kParts + p) * 2 + kb; a database
// tile is one row block.
template <typename ROW, int QTILE, int STAGES>
struct ScanShape {
  using Row = ROW;
  static constexpr bool kSplit = std::is_same<ROW, float>::value;
  static constexpr int kQTile = QTILE, kStages = STAGES;
  static constexpr int kParts = kSplit ? 2 : 1, kCols = kParts * kHidden;
  static constexpr int kRowBlocks = QTILE / 128;
  static constexpr int kTerms = kSplit ? 3 : 1;     // MMAs per K step: hi.hi [, hi.lo, lo.hi]
  static constexpr int kQBoxes = kRowBlocks * kParts * 2, kDbBoxes = kParts * 2;
  static constexpr int kQBytes = kQBoxes * kBoxBytes, kDbBytes = kDbBoxes * kBoxBytes;
  static constexpr int kAccCols = kRowBlocks * 128; // TMEM columns of one of the two accumulators
  static constexpr int kEpiWarps = QTILE / 32, kMmaWarp = kEpiWarps, kLoadWarp = kEpiWarps + 1,
                       kWarps = kEpiWarps + 2;
  // barriers
  static constexpr int kBarQFull = 0, kBarQEmpty = 1, kBarBFull = 2, kBarBEmpty = kBarBFull + STAGES,
                       kBarDFull = kBarBEmpty + STAGES, kBarDEmpty = kBarDFull + 2, kNumBars = kBarDEmpty + 2;
  // dynamic shared memory
  static constexpr int off_q = 0;
  static constexpr int off_db = off_q + kQBytes;
  static constexpr int off_d2 = off_db + STAGES * kDbBytes;
  static constexpr int off_bar = off_d2 + kD2Slots * kDbTile * 4;
  static constexpr int off_tmem = off_bar + kNumBars * 8;
  static constexpr int off_list = (off_tmem + 8 + 15) & ~15;
  static constexpr int smem_bytes(int kc) { return off_list + kc * QTILE * 8; }   // per-thread sorted lists
};

// Certificate margin of the fp16 scan, relative: eps = 2^-14 |q| N_max (cosine) or
// 2^-14 (2 |q| N_max + N_max^2 + |q|^2) (L2, the scan's frame), N_max the
// largest row norm.  It has to cover the exact chain's error plus the tensor
// cores' error on the same dot product.  The sequential chain of 128 FMAs is
// within 128 * 2^-24 * sum|q_i x_i| = 2^-17 sum|q_i x_i| of the real value.
// Published measurements of fp16-input, fp32-accumulate tensor cores on earlier
// NVIDIA generations show an accumulator that truncates, about 2^-23 per
// addition, which over 128 products is 2^-16 sum|q_i x_i|; and
// sum|q_i x_i| <= |q| N_max (for L2 the terms of 2 q.d - |d|^2 and |q|^2 add
// the other two parts).  2^-14 leaves a margin of at least 4x over the sum.
// The B200's accumulator has not been measured: this constant rests on that
// argument, not on a measurement.
struct F16Scan : ScanShape<__half, 256, 3> {
  static constexpr float kCertRel = 1.f / 16384.f;
};

// Certificate margin of the split scan:
//   cosine  eps = kCertRel |q| N_max + kCertAbs (|q| + N_max)
//   L2      eps = kCertRel (2 |q| N_max + N_max^2 + |q|^2) + 2 kCertAbs (|q| + N_max)
// (the scan's frame, as F16Scan).  Against the real dot product R = sum q_i x_i:
//  * the split.  With fp16 hi and lo normal, q_i = qh_i + ql_i + e_i, |e_i| <= 2^-22 |q_i|
//    (hi is within 2^-11 |q_i|, lo within 2^-11 of the rest), and the same for x.  The scan
//    sums qh.xh + qh.xl + ql.xh = (q - e_q).(x - e_x) - ql.xl; with |ql_i| <= 2^-11 (1 + 2^-11)
//    |q_i| that is within (3 + 2^-9) 2^-22 < 2^-20 of sum |q_i x_i| from R, the dropped lo.lo
//    term included;
//  * subnormals.  Where x_i - hi_i (or x_i itself) is below 2^-14, lo (or hi) is rounded onto
//    the fp16 subnormal grid of spacing 2^-24: an absolute error of at most 2^-25 per
//    component, which sums to 2^-25 (|q|_1 + |x|_1) <= 2^-25 sqrt(128) (|q| + N_max)
//    < 2^-21 (|q| + N_max) = kCertAbs (|q| + N_max).  This assumes that kind::f16 takes
//    subnormal fp16 operands at their value; an MMA that flushed them would lose up to 2^-14
//    per component;
//  * the tensor-core accumulator.  3 x 128 products go into one fp32 accumulator; on the
//    truncation argument of F16Scan (about 2^-23 per addition) that is within
//    384 x 2^-23 (1 + 2^-10) < 2^-14.4 of sum |q_i x_i|;
//  * the exact chain: within 2^-17 sum |q_i x_i| (F16Scan).  For L2 the fp32 difference
//    q_i - x_i adds 2^-23 relative per term of sum (q_i - x_i)^2 <= (|q| + N_max)^2.
// The sum is below 2^-14.1 sum |q_i x_i| <= 2^-14.1 |q| N_max; 2^-13 leaves more than 2x
// (for L2, 2 q.d doubles the first and the |d|^2, |q|^2 and chain errors, each <= 2^-16.9 of
// their square, stay inside the other terms).  As for F16Scan, the B200's accumulator has not
// been measured: this margin rests on the argument, not on a measurement.  Without the split
// (a scan of fp16(x) only) the rounding of the inputs alone is 2^-11 sum |q_i x_i| per side.
struct SplitScan : ScanShape<float, 128, 2> {
  static constexpr float kCertRel = 1.f / 8192.f, kCertAbs = 1.f / 2097152.f;
};

static_assert(F16Scan::smem_bytes(kMaxCand) <= 232448, "exceeds the 227 KB shared-memory limit of sm_100");
static_assert(SplitScan::smem_bytes(kMaxCand) <= 232448, "exceeds the 227 KB shared-memory limit of sm_100");

struct alignas(64) Maps {
  CUtensorMap q, db;
};

// Workspace header: the int64 count of queries that took the exact fallback in
// the last call (read by EmbeddingIndex.last_fallbacks), then the largest
// squared row norm (float bits; atomicMax on the bits orders non-negative
// floats).  Zeroed by every call.
constexpr size_t kOffFallbacks = 0, kOffMaxSqNorm = 8, kHeaderBytes = 256;

struct Plan {
  int64_t tiles_q, tiles_db, segs, tiles_per_seg, qp;
  int kc;
  int64_t sample_tiles;       // 0 = no seeding pre-pass
  size_t off_flagged, off_scores, off_index, off_d2, off_seed_scores, off_seed_index, total;
  size_t off_qimage;          // split scan: [Q, 256] hi | lo image of the queries
};

template <class Cfg>
static Plan make_plan(int64_t Q, int64_t D, int k) {
  Plan p{};
  p.tiles_q = (Q + Cfg::kQTile - 1) / Cfg::kQTile;
  p.tiles_db = (D + kDbTile - 1) / kDbTile;
  p.qp = p.tiles_q * Cfg::kQTile;
  int64_t segs = 1;
  if (p.tiles_q > 0 && p.tiles_q < int64_t(kWaves) * kNumSMs)
    segs = (int64_t(kWaves) * kNumSMs + p.tiles_q - 1) / p.tiles_q;
  const int64_t max_segs = p.tiles_db / 16 > 1 ? p.tiles_db / 16 : 1;   // >= 16 tiles per segment
  if (segs > max_segs) segs = max_segs;
  p.tiles_per_seg = p.tiles_db > 0 ? (p.tiles_db + segs - 1) / segs : 1;
  p.segs = p.tiles_db > 0 ? (p.tiles_db + p.tiles_per_seg - 1) / p.tiles_per_seg : 1;
  int kc = (k + 4 + 3) & ~3;
  p.kc = kc > kMaxCand ? kMaxCand : kc;
  auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
  const size_t cand = size_t(p.segs) * p.qp * p.kc;
  p.off_flagged = kHeaderBytes;                              // [Q] int32 queries to rescan
  p.off_scores = p.off_flagged + up(size_t(Q) * 4);
  p.off_index = p.off_scores + up(cand * 4);
  p.off_d2 = p.off_index + up(cand * 4);
  p.total = p.off_d2 + up(size_t(p.tiles_db) * kDbTile * 4);
  // Seeding pays when the sample is a small part of the scan.
  p.sample_tiles = p.tiles_db >= 8 * kSampleTiles ? kSampleTiles : 0;
  p.off_seed_scores = p.total;
  p.off_seed_index = p.off_seed_scores + up(size_t(p.qp) * p.kc * 4);
  if (p.sample_tiles) p.total = p.off_seed_index + up(size_t(p.qp) * p.kc * 4);
  if (Cfg::kSplit) {
    p.off_qimage = p.total;
    p.total += up(size_t(Q) * Cfg::kCols * 2);
  }
  return p;
}

struct Args {
  const float *d2;            // [tiles_db * 128] squared row norms, +inf past the end (read by the L2 scan)
  float *part_scores;         // [segs][qp][kc]
  int32_t *part_index;
  int64_t tiles_q, tiles_db, segs, tiles_per_seg, qp, num_rows;
  int kc;
  // [qp][kc] lists of a pre-pass over the first kSampleTiles tiles, or NULL.  The
  // kc-th best score of ANY subset of the database is a lower bound of the
  // kc-th best overall, so a scan may start from it instead of -inf: it skips
  // the warm-up in which every value is inserted.
  const float *seed;
};

// Insert (v, idx) into the thread's descending list (column `ls`/`li`, stride
// STRIDE = the scan's query tile).  Strict comparisons: among equal scores the
// earlier (lower) index stays ahead.  Returns the new threshold (the list's last
// score).  (An unsorted set with a tracked eviction slot was tried: its full
// rescan per insert costs more than the average shift here.)
template <int STRIDE>
__device__ __noinline__ float list_insert(float *ls, int32_t *li, int kc, float v, int32_t idx) {
  int j = kc - 1;
  while (j > 0 && ls[(j - 1) * STRIDE] < v) {
    ls[j * STRIDE] = ls[(j - 1) * STRIDE];
    li[j * STRIDE] = li[(j - 1) * STRIDE];
    --j;
  }
  ls[j * STRIDE] = v;
  li[j * STRIDE] = idx;
  return ls[(kc - 1) * STRIDE];
}

// Threshold a scan starts from, given the kc-th score of the seeding sample:
// strictly below it, so rows that tie with the seed still enter.
__device__ __forceinline__ float seed_threshold(float s) { return s - (fabsf(s) * 2.4e-7f + 1e-30f); }

__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// The scan, for the entry points below.
template <class Cfg, int METRIC>
__device__ __forceinline__ void scan(const Maps &maps, const Args &p) {
  using L = Cfg;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *qs = smem + L::off_q, *dbs = smem + L::off_db;
  float *d2s = reinterpret_cast<float *>(smem + L::off_d2);
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::off_bar);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + L::off_tmem);
  float *list_s = reinterpret_cast<float *>(smem + L::off_list);

  // The entry point's __launch_bounds__ bounds threadIdx.x only inside the kernel's
  // own body; stated here too, the warp-role arithmetic compiles as it would there.
  __builtin_assume(threadIdx.x < L::kWarps * 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == L::kMmaWarp) {
    tmem_alloc(tmem_slot, 2 * L::kAccCols);
  } else if (tid == 0) {
    mbar_init(bar + L::kBarQFull, 1);
    mbar_init(bar + L::kBarQEmpty, 1);
    for (int s = 0; s < L::kStages; ++s) {
      mbar_init(bar + L::kBarBFull + s, 1);
      mbar_init(bar + L::kBarBEmpty + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar + L::kBarDFull + a, 1);
      mbar_init(bar + L::kBarDEmpty + a, L::kEpiWarps);
    }
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int64_t items = p.tiles_q * p.segs;

  if (warp == L::kLoadWarp) {
    // ================================ TMA loader =================================
    // (whole warp in the loop, one elected lane issues: see the MMA issuer below)
    uint32_t elected;
    asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(elected));
    const bool issuer = elected != 0u;
    if (issuer) {
      prefetch_tmap(&maps.q);
      prefetch_tmap(&maps.db);
    }
    uint32_t it = 0, item_n = 0;
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x, ++item_n) {
      const int64_t qt = item % p.tiles_q, seg = item / p.tiles_q;
      mbar_wait(bar + L::kBarQEmpty, (item_n & 1) ^ 1);
      if (issuer) {
        mbar_arrive_expect_tx(bar + L::kBarQFull, L::kQBytes);
#pragma unroll
        for (int b = 0; b < L::kQBoxes; ++b) {        // b = (rb * kParts + p) * 2 + kb
          const int rb = b / (2 * L::kParts), pk = b % (2 * L::kParts);
          tma_load_2d(qs + b * kBoxBytes, &maps.q, pk * 64, int(qt * L::kQTile + rb * 128),
                      bar + L::kBarQFull);
        }
      }
      __syncwarp();
      const int64_t t0 = seg * p.tiles_per_seg;
      const int64_t t1 = t0 + p.tiles_per_seg < p.tiles_db ? t0 + p.tiles_per_seg : p.tiles_db;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const uint32_t s = it % L::kStages, ph = (it / L::kStages) & 1;
        uint8_t *dst = dbs + s * L::kDbBytes;
        mbar_wait(bar + L::kBarBEmpty + s, ph ^ 1);
        if (issuer) {
          mbar_arrive_expect_tx(bar + L::kBarBFull + s, L::kDbBytes + (METRIC == 1 ? kDbTile * 4 : 0));
#pragma unroll
          for (int b = 0; b < L::kDbBoxes; ++b)
            tma_load_2d(dst + b * kBoxBytes, &maps.db, b * 64, int(t * kDbTile), bar + L::kBarBFull + s);
          if (METRIC == 1)
            bulk_g2s(d2s + (it % kD2Slots) * kDbTile, p.d2 + t * kDbTile, kDbTile * 4,
                     bar + L::kBarBFull + s);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else if (warp == L::kMmaWarp) {
    // ================================ MMA issuer =================================
    // The whole warp runs the loop and waits on the barriers; one elected lane issues.  Issued
    // from inside `if (lane == 0)` the operands of every MMA were ordinary registers to the
    // compiler and each tcgen05.mma came wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop
    // (11-13 instructions per MMA on a warp that shares its scheduler with epilogue warps: more
    // than the 64 cycles an MMA of this shape takes); with warp-uniform operands they live in
    // uniform registers (measured on the fused layer kernel, DESIGN.md section 9.1).
    constexpr uint32_t idesc = idesc_f16(128, kDbTile);
    const uint32_t qa = smem_u32(qs), ba = smem_u32(dbs);
    const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
    uint32_t elected;
    asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(elected));
    const bool issuer = elected != 0u;
    uint32_t it = 0, item_n = 0;
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x, ++item_n) {
      const int64_t seg = item / p.tiles_q;
      const int64_t t0 = seg * p.tiles_per_seg;
      const int64_t t1 = t0 + p.tiles_per_seg < p.tiles_db ? t0 + p.tiles_per_seg : p.tiles_db;
      mbar_wait(bar + L::kBarQFull, item_n & 1);
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const uint32_t s = it % L::kStages, ph = (it / L::kStages) & 1, a = it & 1, pha = (it >> 1) & 1;
        mbar_wait(bar + L::kBarBFull + s, ph);
        mbar_wait(bar + L::kBarDEmpty + a, pha ^ 1);
        tc_fence_after();
        if (issuer) {
#pragma unroll
          for (int rb = 0; rb < L::kRowBlocks; ++rb) {
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              const int kb = kk >> 2, k = kk & 3;
#pragma unroll
              for (int term = 0; term < L::kTerms; ++term) {   // hi.hi, hi.lo, lo.hi
                const int qpart = term == 2, dpart = term == 1;
                const uint64_t da = smem_desc_sw128(qa + ((rb * L::kParts + qpart) * 2 + kb) * kBoxBytes + k * 32);
                const uint64_t db = smem_desc_sw128(ba + s * L::kDbBytes + (dpart * 2 + kb) * kBoxBytes + k * 32);
                mma_f16_ss(tm + a * L::kAccCols + rb * 128, da, db, idesc, (kk | term) != 0);
              }
            }
          }
          mma_commit(bar + L::kBarBEmpty + s);
          mma_commit(bar + L::kBarDFull + a);
        }
        __syncwarp();
      }
      if (issuer) mma_commit(bar + L::kBarQEmpty);   // every MMA reading this item's queries is done
      __syncwarp();
    }
    __syncwarp();
  } else {
    // ============ epilogue: running top-k, one query per thread ====================
    // A warp reads TMEM lanes 32 (warp % 4) .. +31 (the tcgen05 lane-access rule);
    // with two row blocks, warps 4-7 take the second one's columns.
    const int quad = warp & 3, half = warp >> 2;
    const int row = half * 128 + quad * 32 + lane;          // query inside the item
    const uint32_t tbase = tmem + (uint32_t(quad * 32) << 16) + half * 128;
    const int kc = p.kc;
    const int32_t rows = int32_t(p.num_rows);
    float *ls = list_s + tid;
    int32_t *li = reinterpret_cast<int32_t *>(list_s + kc * L::kQTile) + tid;
    const float ninf = -INFINITY;
    uint32_t it = 0;
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
      const int64_t qt = item % p.tiles_q, seg = item / p.tiles_q;
      const int64_t t0 = seg * p.tiles_per_seg;
      const int64_t t1 = t0 + p.tiles_per_seg < p.tiles_db ? t0 + p.tiles_per_seg : p.tiles_db;
      for (int j = 0; j < kc; ++j) {
        ls[j * L::kQTile] = ninf;
        li[j * L::kQTile] = INT_MAX;
      }
      float seed = ninf;
      if (p.seed)                                   // kc-th best of the sample (lists are sorted)
        seed = seed_threshold(p.seed[(size_t(qt) * L::kQTile + row) * kc + kc - 1]);
      float thr = seed;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const uint32_t a = it & 1, pha = (it >> 1) & 1;
        mbar_wait(bar + L::kBarDFull + a, pha);
        tc_fence_after();
        float v[kDbTile];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) tmem_ld32(tbase + a * L::kAccCols + cb * 32, v + cb * 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + L::kBarDEmpty + a);   // accumulator is in registers now
        const int32_t base = int32_t(t * kDbTile);
        if (METRIC == 1) {
          // -|q-d|^2 = 2 q.d - |d|^2 - |q|^2 ; the last term is constant per query
          const float4 *d2 = reinterpret_cast<const float4 *>(d2s + (it % kD2Slots) * kDbTile);
#pragma unroll
          for (int c4 = 0; c4 < kDbTile / 4; ++c4) {
            const float4 n = d2[c4];
            v[4 * c4] = fmaf(2.f, v[4 * c4], -n.x);
            v[4 * c4 + 1] = fmaf(2.f, v[4 * c4 + 1], -n.y);
            v[4 * c4 + 2] = fmaf(2.f, v[4 * c4 + 2], -n.z);
            v[4 * c4 + 3] = fmaf(2.f, v[4 * c4 + 3], -n.w);
          }
        }
        // hot path: the maximum of the 128 scores as four independent chains of
        // 3-input maxima.  (Rows past the end of the database -- zero-filled by
        // TMA -- may raise it in the last tile; offer() drops them by index.)
        float t4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          t4[q] = fmaxf(v[32 * q], v[32 * q + 1]);
#pragma unroll
          for (int c = 2; c < 32; c += 2) t4[q] = max3(t4[q], v[32 * q + c], v[32 * q + c + 1]);
        }
        const float top = fmaxf(fmaxf(t4[0], t4[1]), fmaxf(t4[2], t4[3]));
        if (top > thr) {
          // rare once the list has warmed up: find the values above the threshold
#pragma unroll
          for (int g = 0; g < kDbTile / 8; ++g) {
            const float gm = fmaxf(max3(v[8 * g], v[8 * g + 1], v[8 * g + 2]),
                                   max3(v[8 * g + 3], v[8 * g + 4],
                                        max3(v[8 * g + 5], v[8 * g + 6], v[8 * g + 7])));
            if (gm > thr) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (v[8 * g + j] > thr && base + 8 * g + j < rows)
                  thr = fmaxf(seed, list_insert<L::kQTile>(ls, li, kc, v[8 * g + j], base + 8 * g + j));
            }
          }
        }
      }
      // hand the segment's candidates to the finish kernel
      const size_t out = (size_t(seg) * p.qp + size_t(qt) * L::kQTile + row) * kc;
      for (int j = 0; j < kc; ++j) {
        p.part_scores[out + j] = ls[j * L::kQTile];
        p.part_index[out + j] = li[j * L::kQTile];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == L::kMmaWarp) tmem_dealloc(tmem, 2 * L::kAccCols);
}

// One kernel per row type; each __launch_bounds__ gives ptxas the register limit
// of that configuration's warp count.
template <int METRIC>
__global__ void __launch_bounds__(F16Scan::kWarps * 32, 1)
topk_scan_kernel(const __grid_constant__ Maps maps, const Args p) {
  scan<F16Scan, METRIC>(maps, p);
}

template <int METRIC>
__global__ void __launch_bounds__(SplitScan::kWarps * 32, 1)
split_search_kernel(const __grid_constant__ Maps maps, const Args p) {
  scan<SplitScan, METRIC>(maps, p);
}

// ---- loads of row components as fp32 ------------------------------------------------
// 16 bytes: 8 fp16 or 4 fp32 components.  (Both forms become the same read-only
// LDG.128; they differ in how far ptxas unrolls the row-norm pass around them,
// and each keeps the unrolling measured with it.)
__device__ __forceinline__ void load_f32(const __half *p, float (&x)[8]) {
  const uint4 raw = *reinterpret_cast<const uint4 *>(p);
  const __half2 *h = reinterpret_cast<const __half2 *>(&raw);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __half22float2(h[j]);
    x[2 * j] = f.x;
    x[2 * j + 1] = f.y;
  }
}
__device__ __forceinline__ void load_f32(const float *p, float (&x)[4]) {
  const float4 v = __ldg(reinterpret_cast<const float4 *>(p));
  x[0] = v.x;
  x[1] = v.y;
  x[2] = v.z;
  x[3] = v.w;
}
// 4 fp16 components (a lane's quarter of a query), 2 bytes at a time
__device__ __forceinline__ void load_f32(const __half *p, float (&x)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) x[j] = __half2float(p[j]);
}

// components of a row per 16-byte load
template <typename Row>
constexpr int kChunk = 16 / int(sizeof(Row));

// ---- |d|^2 per database row (L2 metric); +inf for the padding rows; and the ----------
// largest |d|^2 of the real rows into *max_sqnorm (float bits, zeroed by the caller)
template <typename Row>
__global__ void __launch_bounds__(256)
row_sqnorm_kernel(const Row *__restrict__ db, int64_t rows, int64_t padded, float *__restrict__ out,
                  unsigned int *__restrict__ max_sqnorm) {
  constexpr int n = kChunk<Row>;
  const int sub = threadIdx.x & 15;
  const int64_t per_pass = int64_t(gridDim.x) * (blockDim.x >> 4);
  float top = 0.f;
  for (int64_t i = int64_t(blockIdx.x) * (blockDim.x >> 4) + (threadIdx.x >> 4); i < padded;
       i += per_pass) {
    float s = 0.f;
    if (i < rows) {
#pragma unroll
      for (int c = 0; c < 8; c += n) {
        float x[n];
        load_f32(db + i * kHidden + sub * 8 + c, x);
#pragma unroll
        for (int j = 0; j < n; ++j) s = fmaf(x[j], x[j], s);
      }
    }
#pragma unroll
    for (int d = 8; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d, 16);
    if (sub == 0) out[i] = i < rows ? s : INFINITY;
    if (i < rows) top = fmaxf(top, s);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) top = fmaxf(top, __shfl_xor_sync(0xffffffffu, top, d));
  if ((threadIdx.x & 31) == 0) atomicMax(max_sqnorm, __float_as_uint(top));
}

// ---- ordering -----------------------------------------------------------------------
// (score desc, index asc).  `better(a, b)`: a sorts before b.
template <typename I>
__device__ __forceinline__ bool better(float sa, I ia, float sb, I ib) {
  return sa > sb || (sa == sb && ia < ib);
}

template <typename I>
__device__ __forceinline__ void warp_best(float &s, I &i) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const float so = __shfl_xor_sync(0xffffffffu, s, d);
    const I io = __shfl_xor_sync(0xffffffffu, i, d);
    if (better<I>(so, io, s, i)) {
      s = so;
      i = io;
    }
  }
}

// One step of the exact score's chain: the finish and the fallback passes share
// it, so they produce the same bits.
template <int METRIC>
__device__ __forceinline__ float exact_step(float acc, float q, float x) {
  if (METRIC == 0) return fmaf(q, x, acc);
  const float d = q - x;
  return fmaf(d, d, acc);
}

// Exact score of (query in shared memory as fp32, database row): a sequential
// fp32 FMA chain in dimension order.
template <int METRIC, typename Row>
__device__ __forceinline__ float exact_score(const float *q, const Row *row) {
  constexpr int n = kChunk<Row>;
  float acc = 0.f;
#pragma unroll 4
  for (int c = 0; c < kHidden / n; ++c) {
    float x[n];
    load_f32(row + c * n, x);
#pragma unroll
    for (int j = 0; j < n; ++j) acc = exact_step<METRIC>(acc, q[c * n + j], x[j]);
  }
  return METRIC == 0 ? acc : -acc;
}

constexpr int kFinishWarps = 4;

// k selection rounds over the (score desc, index asc) order of query qi's
// segs x kc candidate slots (index INT_MAX = empty slot).  Writes the output
// row; returns the k-th score, or -inf when fewer than k rows exist.  One warp.
__device__ __forceinline__ float select_topk(const float *__restrict__ part_scores, const int32_t *__restrict__ part_index,
                             int64_t segs, int64_t qp, int kc, int64_t qi, int k, int64_t index_base,
                             float *__restrict__ out_scores, int64_t *__restrict__ out_index) {
  const int lane = threadIdx.x & 31;
  const int64_t C = segs * kc;
  float last_s = INFINITY;
  int32_t last_i = -1;
  for (int r = 0; r < k; ++r) {
    float bs = -INFINITY;
    int32_t bi = INT_MAX;
    for (int64_t c = lane; c < C; c += 32) {
      const size_t off = (size_t(c / kc) * qp + qi) * kc + (c % kc);
      const int32_t i = part_index[off];
      const float s = part_scores[off];
      if (i != INT_MAX && better<int32_t>(last_s, last_i, s, i) && better<int32_t>(s, i, bs, bi)) {
        bs = s;
        bi = i;
      }
    }
    warp_best<int32_t>(bs, bi);
    if (lane == 0) {
      out_scores[qi * k + r] = bi == INT_MAX ? -INFINITY : bs;
      out_index[qi * k + r] = bi == INT_MAX ? int64_t(-1) : index_base + bi;
    }
    if (bi == INT_MAX) {             // fewer than k rows exist: pad the tail
      for (int rr = r + 1 + lane; rr < k; rr += 32) {
        out_scores[qi * k + rr] = -INFINITY;
        out_index[qi * k + rr] = -1;
      }
      return -INFINITY;
    }
    last_s = bs;
    last_i = bi;
  }
  return last_s;
}

// One warp per query: exact rescoring of the candidates, selection, and the
// certificate.  `seed` is the seeding pre-pass's [qp][kc] lists or NULL;
// uncertified queries are appended to `flagged` (count in *fallbacks).  For fp32
// rows a query with a component above the fp16 range (its hi part is inf; the
// scan's scores for it are meaningless) is flagged whatever its certificate.
template <class Cfg, int METRIC>
__global__ void __launch_bounds__(kFinishWarps * 32)
topk_finish_kernel(const typename Cfg::Row *__restrict__ queries, const typename Cfg::Row *__restrict__ db,
                   float *__restrict__ part_scores, const int32_t *__restrict__ part_index,
                   const float *__restrict__ seed, const unsigned int *__restrict__ max_sqnorm,
                   int64_t segs, int64_t qp, int kc, int64_t Q, int k, int64_t index_base,
                   float *__restrict__ out_scores, int64_t *__restrict__ out_index,
                   unsigned long long *__restrict__ fallbacks, int32_t *__restrict__ flagged) {
  __shared__ float qsm[kFinishWarps][kHidden];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t qi = int64_t(blockIdx.x) * kFinishWarps + warp;
  if (qi >= Q) return;
  float *q = qsm[warp];
  float v[4];
  load_f32(queries + qi * kHidden + lane * 4, v);
#pragma unroll
  for (int j = 0; j < 4; ++j) q[lane * 4 + j] = v[j];
  // |q|^2 sets eps to its last bit, and so which borderline queries are
  // certified: each row type keeps its own order of the sum.
  float qq = 0.f, qmax = 0.f;
  if constexpr (Cfg::kSplit) {
    qq = fmaf(v[0], v[0], fmaf(v[1], v[1], fmaf(v[2], v[2], fmaf(v[3], v[3], qq))));
    qmax = fmaxf(fmaxf(fabsf(v[0]), fabsf(v[1])), fmaxf(fabsf(v[2]), fabsf(v[3])));
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) qq = fmaf(v[j], v[j], qq);
  }
  // pass 0, before the tensor-core scores are overwritten: every row the scan
  // dropped has a tensor-core score <= max(seed', last entry of a full list)
  float bound = seed ? seed_threshold(seed[qi * kc + kc - 1]) : -INFINITY;
  for (int64_t s = lane; s < segs; s += 32) {
    const size_t off = (size_t(s) * qp + qi) * kc + kc - 1;
    if (part_index[off] != INT_MAX) bound = fmaxf(bound, part_scores[off]);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    qq += __shfl_xor_sync(0xffffffffu, qq, d);
    if constexpr (Cfg::kSplit) qmax = fmaxf(qmax, __shfl_xor_sync(0xffffffffu, qmax, d));
    bound = fmaxf(bound, __shfl_xor_sync(0xffffffffu, bound, d));
  }
  __syncwarp();
  const int64_t C = segs * kc;
  // pass 1: exact scores, written over the tensor-core scores
  for (int64_t c = lane; c < C; c += 32) {
    const size_t off = (size_t(c / kc) * qp + qi) * kc + (c % kc);
    const int32_t idx = part_index[off];
    part_scores[off] = idx == INT_MAX ? -INFINITY : exact_score<METRIC>(q, db + int64_t(idx) * kHidden);
  }
  __syncwarp();
  // pass 2: selection
  const float sk = select_topk(part_scores, part_index, segs, qp, kc, qi, k, index_base, out_scores,
                               out_index);
  // certificate: no dropped row can reach the k-th exact score (the Cfg's margin).
  // A query whose scan dropped nothing (B = -inf: small databases) is exact as it is.
  const float n2 = __uint_as_float(*max_sqnorm), qn = sqrtf(qq), nmax = sqrtf(n2);
  float eps = METRIC == 0 ? Cfg::kCertRel * qn * nmax : Cfg::kCertRel * (2.f * qn * nmax + n2 + qq);
  if constexpr (Cfg::kSplit) {
    const float abs_eps = Cfg::kCertAbs * (qn + nmax);
    eps += METRIC == 0 ? abs_eps : 2.f * abs_eps;
  }
  const float sk_scan = METRIC == 0 ? sk : sk + qq;
  // (For fp16 rows the compiler fuses `bound + eps` with eps's last product: rewriting
  // these lines can move that rounding, and with it last_fallbacks().)
  bool flag = bound > -INFINITY && !(bound + eps < sk_scan);
  if constexpr (Cfg::kSplit) flag = !(qmax <= 65504.f) || flag;
  if (lane == 0 && flag) flagged[atomicAdd(fallbacks, 1ull)] = int32_t(qi);
}

// ---- exact fallback -----------------------------------------------------------------
// Work item = (group of kFbWarps flagged queries, database segment): the CTA
// stages 64 rows at a time in shared memory as fp32 (read from global memory
// once for the whole group); warp w scores them for query w with the exact
// chain (two rows per lane) and keeps the segment's k best by (score desc,
// index asc) in registers, entry j in lane j.  The list goes to the query's
// candidate slots of that segment (the first k of kc; the rest emptied), which
// topk_fallback_select_kernel then reduces as the finish kernel does.
constexpr int kFbWarps = 8, kFbRows = 64, kFbStride = kHidden + 1;   // +1: conflict-free columns
constexpr int kFbBlocksPerSM = 4;

// Rows [t, min(t + kFbRows, r1)) of the database into xs as fp32, zeros past r1.
__device__ __forceinline__ void stage_rows(float *xs, const __half *db, int64_t t, int64_t r1) {
  for (int e = threadIdx.x; e < kFbRows * (kHidden / 8); e += kFbWarps * 32) {
    const int r = e / (kHidden / 8), c = e % (kHidden / 8);
    float x[8] = {};
    if (t + r < r1) load_f32(db + (t + r) * kHidden + c * 8, x);
#pragma unroll
    for (int j = 0; j < 8; ++j) xs[r * kFbStride + c * 8 + j] = x[j];
  }
}
__device__ __forceinline__ void stage_rows(float *xs, const float *db, int64_t t, int64_t r1) {
#pragma unroll 1   // unrolled, ptxas spills at 48 registers
  for (int e = threadIdx.x; e < kFbRows * (kHidden / 4); e += kFbWarps * 32) {
    const int r = e / (kHidden / 4), c = e % (kHidden / 4);
    float x[4] = {};
    if (t + r < r1) load_f32(db + (t + r) * kHidden + c * 4, x);
#pragma unroll
    for (int j = 0; j < 4; ++j) xs[r * kFbStride + c * 4 + j] = x[j];
  }
}

template <class Cfg, int METRIC>
__global__ void __launch_bounds__(kFbWarps * 32)
topk_fallback_scan_kernel(const typename Cfg::Row *__restrict__ queries, const typename Cfg::Row *__restrict__ db,
                          int64_t num_rows, int64_t rows_per_seg, int64_t segs, int64_t qp, int kc, int k,
                          const unsigned long long *__restrict__ fallbacks,
                          const int32_t *__restrict__ flagged, float *__restrict__ part_scores,
                          int32_t *__restrict__ part_index) {
  __shared__ float xs[kFbRows * kFbStride];
  __shared__ float qsm[kFbWarps][kHidden];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n = int64_t(*fallbacks);
  const int64_t groups = (n + kFbWarps - 1) / kFbWarps;
  for (int64_t w = blockIdx.x; w < groups * segs; w += gridDim.x) {
    const int64_t g = w % groups, seg = w / groups;     // neighbouring CTAs share a segment (L2)
    const bool active = g * kFbWarps + warp < n;        // warp-uniform
    const int64_t qi = active ? flagged[g * kFbWarps + warp] : 0;
    __syncthreads();                                    // the previous item is done with qsm / xs
    if (active) {
      float v[4];
      load_f32(queries + qi * kHidden + lane * 4, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) qsm[warp][lane * 4 + j] = v[j];
    }
    const float *q = qsm[warp];
    float ls = -INFINITY, ts = -INFINITY;               // this lane's entry; the k-th entry
    int32_t li = INT_MAX, ti = INT_MAX;
    const int64_t r0 = seg * rows_per_seg;
    const int64_t r1 = r0 + rows_per_seg < num_rows ? r0 + rows_per_seg : num_rows;
    for (int64_t t = r0; t < r1; t += kFbRows) {
      __syncthreads();
      stage_rows(xs, db, t, r1);
      __syncthreads();
      if (!active) continue;
      const float *x0 = xs + lane * kFbStride, *x1 = xs + (lane + 32) * kFbStride;
      float a0 = 0.f, a1 = 0.f;
#pragma unroll 16
      for (int d = 0; d < kHidden; ++d) {
        a0 = exact_step<METRIC>(a0, q[d], x0[d]);
        a1 = exact_step<METRIC>(a1, q[d], x1[d]);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float s = METRIC == 0 ? (h ? a1 : a0) : -(h ? a1 : a0);
        const int32_t i = int32_t(t + h * 32 + lane);
        unsigned int m = __ballot_sync(0xffffffffu, t + h * 32 + lane < r1 && better<int32_t>(s, i, ts, ti));
        while (m) {                                     // rare once the list has filled
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const float cs = __shfl_sync(0xffffffffu, s, src);
          const int32_t ci = __shfl_sync(0xffffffffu, i, src);
          if (!better<int32_t>(cs, ci, ts, ti)) continue;
          const int pos = __popc(__ballot_sync(0xffffffffu, lane < k && better<int32_t>(ls, li, cs, ci)));
          const float us = __shfl_up_sync(0xffffffffu, ls, 1);
          const int32_t ui = __shfl_up_sync(0xffffffffu, li, 1);
          if (lane > pos) {
            ls = us;
            li = ui;
          } else if (lane == pos) {
            ls = cs;
            li = ci;
          }
          ts = __shfl_sync(0xffffffffu, ls, k - 1);
          ti = __shfl_sync(0xffffffffu, li, k - 1);
        }
      }
    }
    if (active && lane < kc) {
      const size_t off = (size_t(seg) * qp + qi) * kc + lane;
      part_scores[off] = lane < k ? ls : -INFINITY;
      part_index[off] = lane < k ? li : INT_MAX;
    }
  }
}

__global__ void __launch_bounds__(kFinishWarps * 32)
topk_fallback_select_kernel(const float *__restrict__ part_scores, const int32_t *__restrict__ part_index,
                            int64_t segs, int64_t qp, int kc, int k, int64_t index_base,
                            const unsigned long long *__restrict__ fallbacks,
                            const int32_t *__restrict__ flagged, float *__restrict__ out_scores,
                            int64_t *__restrict__ out_index) {
  const int warp = threadIdx.x >> 5;
  const int64_t n = int64_t(*fallbacks);
  for (int64_t f = int64_t(blockIdx.x) * kFinishWarps + warp; f < n; f += int64_t(gridDim.x) * kFinishWarps)
    select_topk(part_scores, part_index, segs, qp, kc, flagged[f], k, index_base, out_scores, out_index);
}

__global__ void __launch_bounds__(kFinishWarps * 32)
topk_merge_kernel(const float *__restrict__ in_scores, const int64_t *__restrict__ in_index, int parts,
                  int64_t Q, int k, float *__restrict__ out_scores, int64_t *__restrict__ out_index) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t qi = int64_t(blockIdx.x) * kFinishWarps + warp;
  if (qi >= Q) return;
  const int C = parts * k;
  const int64_t none = INT64_MAX;
  float last_s = INFINITY;
  int64_t last_i = -1;
  for (int r = 0; r < k; ++r) {
    float bs = -INFINITY;
    int64_t bi = none;
    for (int c = lane; c < C; c += 32) {
      const size_t off = (size_t(c / k) * Q + qi) * k + (c % k);
      const int64_t i = in_index[off];
      const float s = in_scores[off];
      if (i >= 0 && better<int64_t>(last_s, last_i, s, i) && better<int64_t>(s, i, bs, bi)) {
        bs = s;
        bi = i;
      }
    }
    warp_best<int64_t>(bs, bi);
    if (lane == 0) {
      out_scores[qi * k + r] = bi == none ? -INFINITY : bs;
      out_index[qi * k + r] = bi == none ? int64_t(-1) : bi;
    }
    if (bi == none) {
      for (int rr = r + 1 + lane; rr < k; rr += 32) {
        out_scores[qi * k + rr] = -INFINITY;
        out_index[qi * k + rr] = -1;
      }
      break;
    }
    last_s = bs;
    last_i = bi;
  }
}

// [rows, 128] fp32 -> [rows, 256] fp16 image hi | lo, hi = fp16(x), lo = fp16(x - hi)
// (round to nearest; fp16 subnormals kept).  One thread per 4 components.
__global__ void __launch_bounds__(256)
split_rows_kernel(const float *__restrict__ x, int64_t rows, __half *__restrict__ image) {
  const int64_t n = rows * (kHidden / 4);
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = i / (kHidden / 4), c = (i % (kHidden / 4)) * 4;
    const float4 v = __ldg(reinterpret_cast<const float4 *>(x) + i);
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    const float2 b0 = __half22float2(h0), b1 = __half22float2(h1);
    const __half2 l0 = __floats2half2_rn(v.x - b0.x, v.y - b0.y), l1 = __floats2half2_rn(v.z - b1.x, v.w - b1.y);
    __half2 *hi = reinterpret_cast<__half2 *>(image + r * 2 * kHidden + c);
    __half2 *lo = reinterpret_cast<__half2 *>(image + r * 2 * kHidden + kHidden + c);
    hi[0] = h0;
    hi[1] = h1;
    lo[0] = l0;
    lo[1] = l1;
  }
}

static int split_rows(const float *x, int64_t rows, __half *image, cudaStream_t st) {
  int64_t blocks = (rows * (kHidden / 4) + 255) / 256;
  if (blocks > int64_t(kNumSMs) * 16) blocks = int64_t(kNumSMs) * 16;
  split_rows_kernel<<<int(blocks), 256, 0, st>>>(x, rows, image);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

template <class Cfg, int METRIC>
static int launch_scan(const Maps &maps, const Args &a, int64_t items, cudaStream_t st) {
  const auto kernel = Cfg::kSplit ? split_search_kernel<METRIC> : topk_scan_kernel<METRIC>;
  const int smem = Cfg::smem_bytes(a.kc);
  GFX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
  const int grid = int(items < kNumSMs ? items : kNumSMs);
  kernel<<<grid, Cfg::kWarps * 32, smem, st>>>(maps, a);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

// scan (after the optional seeding pre-pass), finish with the certificate, and
// the exact fallback for the flagged queries -- all stream-ordered, no host sync
template <class Cfg, int METRIC>
static int search(const Maps &maps, const Args &a, const Args &pre, const Plan &plan,
                  const typename Cfg::Row *q, const typename Cfg::Row *db, int64_t Q, int64_t num_rows, int k,
                  int64_t index_base, float *out_scores, int64_t *out_index, unsigned long long *fallbacks,
                  const unsigned int *max_sqnorm, int32_t *flagged, cudaStream_t st) {
  int rc = plan.sample_tiles ? launch_scan<Cfg, METRIC>(maps, pre, plan.tiles_q, st) : GFX_OK;
  if (!rc) rc = launch_scan<Cfg, METRIC>(maps, a, plan.tiles_q * plan.segs, st);
  if (rc) return rc;
  const int finish_blocks = int((Q + kFinishWarps - 1) / kFinishWarps);
  topk_finish_kernel<Cfg, METRIC><<<finish_blocks, kFinishWarps * 32, 0, st>>>(
      q, db, a.part_scores, a.part_index, a.seed, max_sqnorm,
      plan.segs, plan.qp, plan.kc, Q, k, index_base, out_scores, out_index, fallbacks, flagged);
  GFX_LAUNCH_CHECK();
  topk_fallback_scan_kernel<Cfg, METRIC><<<kNumSMs * kFbBlocksPerSM, kFbWarps * 32, 0, st>>>(
      q, db, num_rows, plan.tiles_per_seg * kDbTile, plan.segs, plan.qp, plan.kc, k, fallbacks, flagged,
      a.part_scores, a.part_index);
  GFX_LAUNCH_CHECK();
  topk_fallback_select_kernel<<<kNumSMs, kFinishWarps * 32, 0, st>>>(
      a.part_scores, a.part_index, plan.segs, plan.qp, plan.kc, k, index_base, fallbacks, flagged,
      out_scores, out_index);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

// gfx_topk / gfx_topk_f32.  `image` is the database's MMA operand: the rows
// themselves for fp16, their [rows, 256] hi | lo image for fp32.
template <class Cfg>
static int run_search(const char *name, const typename Cfg::Row *queries, int64_t num_queries,
                      const typename Cfg::Row *database, const void *image, int64_t num_rows, int dim, int k,
                      int metric, int64_t index_base, float *out_scores, int64_t *out_index,
                      void *workspace, size_t workspace_bytes, void *stream) {
  const std::string fn(name);
  if (dim != kHidden) return fail(GFX_ERR_UNSUPPORTED, fn + ": kernels are specialised for dim = 128");
  if (k < 1 || k > kMaxK) return fail(GFX_ERR_ARGUMENT, fn + ": k must be in [1, 24]");
  if (metric != 0 && metric != 1) return fail(GFX_ERR_ARGUMENT, fn + ": metric must be 0 (cosine) or 1 (L2)");
  if (num_queries < 0 || num_rows < 0 || num_rows > int64_t(INT_MAX) - 256)
    return fail(GFX_ERR_ARGUMENT, fn + ": bad sizes (rows per call must fit int32)");
  if (num_queries == 0) return GFX_OK;
  if (!queries || !out_scores || !out_index || (num_rows > 0 && (!database || !image)))
    return fail(GFX_ERR_ARGUMENT, fn + ": null pointer");
  if ((reinterpret_cast<uintptr_t>(queries) | reinterpret_cast<uintptr_t>(database) |
       reinterpret_cast<uintptr_t>(image)) & 15)
    return fail(GFX_ERR_ARGUMENT, fn + (Cfg::kSplit ? ": queries, database and image must be 16-byte aligned"
                                                    : ": queries and database must be 16-byte aligned"));
  const Plan plan = make_plan<Cfg>(num_queries, num_rows, k);
  if (workspace_bytes < plan.total || !workspace)
    return fail(GFX_ERR_WORKSPACE, fn + ": workspace too small");
  cudaStream_t st = as_stream(stream);
  char *ws = static_cast<char *>(workspace);
  Args a{};
  a.part_scores = reinterpret_cast<float *>(ws + plan.off_scores);
  a.part_index = reinterpret_cast<int32_t *>(ws + plan.off_index);
  a.d2 = reinterpret_cast<float *>(ws + plan.off_d2);
  a.tiles_q = plan.tiles_q; a.tiles_db = plan.tiles_db; a.segs = plan.segs;
  a.tiles_per_seg = plan.tiles_per_seg; a.qp = plan.qp; a.num_rows = num_rows; a.kc = plan.kc;
  const int finish_blocks = int((num_queries + kFinishWarps - 1) / kFinishWarps);
  // fallback count and largest squared row norm start at 0
  GFX_CUDA(cudaMemsetAsync(ws, 0, kHeaderBytes, st));
  if (num_rows == 0) {
    // empty database: a merge of zero lists writes (-inf, -1) everywhere
    StageScope scope(GFX_STAGE_TOPK, st, 1);
    topk_merge_kernel<<<finish_blocks, kFinishWarps * 32, 0, st>>>(nullptr, nullptr, 0, num_queries, k,
                                                                   out_scores, out_index);
    GFX_LAUNCH_CHECK();
    return GFX_OK;
  }
  __half *qimage = reinterpret_cast<__half *>(ws + plan.off_qimage);   // split scan only
  Maps maps;
  int rc = tma::make_rows_map(&maps.q, Cfg::kSplit ? static_cast<const void *>(qimage) : queries, num_queries,
                              Cfg::kCols, 128);
  if (!rc) rc = tma::make_rows_map(&maps.db, image, num_rows, Cfg::kCols, kDbTile);
  if (rc) return rc;
  // [query split,] sqnorm, [pre-pass,] scan, finish, fallback scan, fallback select
  StageScope scope(GFX_STAGE_TOPK, st, 5 + (Cfg::kSplit ? 1 : 0) + (plan.sample_tiles ? 1 : 0));
  if constexpr (Cfg::kSplit) {
    rc = split_rows(queries, num_queries, qimage, st);
    if (rc) return rc;
  }
  Args pre = a;                            // seeding pre-pass over the first rows, one segment
  if (plan.sample_tiles) {
    pre.part_scores = reinterpret_cast<float *>(ws + plan.off_seed_scores);
    pre.part_index = reinterpret_cast<int32_t *>(ws + plan.off_seed_index);
    pre.tiles_db = pre.tiles_per_seg = plan.sample_tiles;
    pre.segs = 1;
    pre.num_rows = plan.sample_tiles * kDbTile;
    a.seed = pre.part_scores;
  }
  auto *fallbacks = reinterpret_cast<unsigned long long *>(ws + kOffFallbacks);
  auto *max_sqnorm = reinterpret_cast<unsigned int *>(ws + kOffMaxSqNorm);
  auto *flagged = reinterpret_cast<int32_t *>(ws + plan.off_flagged);
  {
    const int64_t padded = plan.tiles_db * kDbTile;
    int64_t blocks = (padded + 15) / 16;
    if (blocks > int64_t(kNumSMs) * 8) blocks = int64_t(kNumSMs) * 8;
    row_sqnorm_kernel<<<int(blocks), 256, 0, st>>>(database, num_rows, padded, const_cast<float *>(a.d2),
                                                   max_sqnorm);
    GFX_LAUNCH_CHECK();
  }
  return metric == 1
      ? search<Cfg, 1>(maps, a, pre, plan, queries, database, num_queries, num_rows, k, index_base, out_scores,
                       out_index, fallbacks, max_sqnorm, flagged, st)
      : search<Cfg, 0>(maps, a, pre, plan, queries, database, num_queries, num_rows, k, index_base, out_scores,
                       out_index, fallbacks, max_sqnorm, flagged, st);
}

}  // namespace topk
}  // namespace gfx

using namespace gfx;

extern "C" size_t gfx_topk_workspace_bytes(int64_t num_queries, int64_t num_rows, int k) {
  if (num_queries <= 0 || num_rows < 0 || k <= 0) return 256;
  return topk::make_plan<topk::F16Scan>(num_queries, num_rows, k).total;
}

extern "C" int gfx_topk(const void *queries, int64_t num_queries, const void *database,
                        int64_t num_rows, int dim, int k, int metric, int64_t index_base,
                        float *out_scores, int64_t *out_index, void *workspace,
                        size_t workspace_bytes, void *stream) {
  const auto *db = static_cast<const __half *>(database);
  return topk::run_search<topk::F16Scan>("gfx_topk", static_cast<const __half *>(queries), num_queries, db, db,
                                         num_rows, dim, k, metric, index_base, out_scores, out_index,
                                         workspace, workspace_bytes, stream);
}

extern "C" int gfx_topk_merge(const float *in_scores, const int64_t *in_index, int parts,
                              int64_t num_queries, int k, float *out_scores, int64_t *out_index,
                              void *stream) {
  if (parts < 0 || k < 1 || num_queries < 0)
    return fail(GFX_ERR_ARGUMENT, "gfx_topk_merge: bad sizes");
  if (num_queries == 0) return GFX_OK;
  if (!out_scores || !out_index || (parts > 0 && (!in_scores || !in_index)))
    return fail(GFX_ERR_ARGUMENT, "gfx_topk_merge: null pointer");
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_TOPK, st, 1);
  const int blocks = int((num_queries + topk::kFinishWarps - 1) / topk::kFinishWarps);
  topk::topk_merge_kernel<<<blocks, topk::kFinishWarps * 32, 0, st>>>(in_scores, in_index, parts,
                                                                     num_queries, k, out_scores, out_index);
  GFX_LAUNCH_CHECK();
  return GFX_OK;
}

extern "C" int gfx_topk_f32_prepare(const float *database, int64_t num_rows, void *image, void *stream) {
  if (num_rows < 0 || num_rows > int64_t(INT_MAX) - 256)
    return fail(GFX_ERR_ARGUMENT, "gfx_topk_f32_prepare: bad sizes (rows per call must fit int32)");
  if (num_rows == 0) return GFX_OK;
  if (!database || !image) return fail(GFX_ERR_ARGUMENT, "gfx_topk_f32_prepare: null pointer");
  if ((reinterpret_cast<uintptr_t>(database) | reinterpret_cast<uintptr_t>(image)) & 15)
    return fail(GFX_ERR_ARGUMENT, "gfx_topk_f32_prepare: database and image must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  StageScope scope(GFX_STAGE_TOPK, st, 1);
  return topk::split_rows(database, num_rows, static_cast<__half *>(image), st);
}

extern "C" size_t gfx_topk_f32_workspace_bytes(int64_t num_queries, int64_t num_rows, int k) {
  if (num_queries <= 0 || num_rows < 0 || k <= 0) return 256;
  return topk::make_plan<topk::SplitScan>(num_queries, num_rows, k).total;
}

extern "C" int gfx_topk_f32(const float *queries, int64_t num_queries, const float *database,
                            const void *image, int64_t num_rows, int dim, int k, int metric,
                            int64_t index_base, float *out_scores, int64_t *out_index, void *workspace,
                            size_t workspace_bytes, void *stream) {
  return topk::run_search<topk::SplitScan>("gfx_topk_f32", queries, num_queries, database, image, num_rows, dim,
                                           k, metric, index_base, out_scores, out_index, workspace,
                                           workspace_bytes, stream);
}
