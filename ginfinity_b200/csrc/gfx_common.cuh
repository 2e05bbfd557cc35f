// Shared declarations for libgfx.so (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <string>
#include <vector>

#include "gfx.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libgfx is written for sm_100a (B200) only"
#endif

namespace gfx {

constexpr int kHidden = 128;  // model.json: hidden = out_dim = 128
constexpr int kMlpHidden = 256;
constexpr int kFeat = 7;
constexpr int kMaxLayers = 8;
constexpr int kMaxEdgeDim = 16;
constexpr int kNumSMs = 148;  // B200

// Row descriptor of the banded fused layer (gfx_row_describe / gfx_edge_describe -> gfx_fused8.cu):
// which of (i-1, type 0) (i+1, type 1) [(partner, type 2|3)] (i-2, type 4) (i+2, type 5) -- the
// reference builder's edge order for nucleotide i (graph.py:494-561) -- the row holds, the partner
// index, or GENERIC when the row is anything else.
namespace rowdesc {
constexpr uint32_t kPrev = 1u, kNext = 2u, kPair = 4u, kPairRev = 8u, kPrev2 = 16u, kNext2 = 32u,
                   kGeneric = 0x80000000u;
constexpr int kPartnerShift = 6, kPartnerBits = 25;
constexpr uint32_t kPartnerMask = (1u << kPartnerBits) - 1u;
}  // namespace rowdesc

void set_error(const std::string &msg);
int fail(int code, const std::string &msg);

#define GFX_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t err__ = (expr);                                               \
    if (err__ != cudaSuccess) {                                               \
      return ::gfx::fail(GFX_ERR_CUDA, std::string(#expr) + ": " +            \
                                           cudaGetErrorString(err__));        \
    }                                                                         \
  } while (0)

#define GFX_LAUNCH_CHECK() GFX_CUDA(cudaGetLastError())

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// gfx_graph.cu: out[i] = sum(in[0..i)); block_sums holds scan_blocks(n) ints;
// *grand_total (optional, device) receives the sum of all n inputs.
int scan_blocks(int64_t n);
int exclusive_scan(const int *in, int *out, int64_t n, int *block_sums, int64_t *grand_total,
                   cudaStream_t st, const int32_t *gate = nullptr);
inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

// Counts `launches` kernel launches for `stage`; if the stage is being
// profiled, brackets the enclosing scope with CUDA events on `st`.
class StageScope {
 public:
  StageScope(int stage, cudaStream_t st, int launches);
  ~StageScope();
  StageScope(const StageScope &) = delete;
  StageScope &operator=(const StageScope &) = delete;

 private:
  cudaStream_t st_;
  cudaEvent_t stop_;
};

}  // namespace gfx

// Host copies of the per-channel vectors: the lean tcgen05 kernels take them
// as kernel parameters (constant bank) instead of loading them on the device.
struct gfx_host_vectors {
  std::vector<float> b1, b2, ln_g, ln_b, ba, bb;
};

// Device-side weights.  One allocation ("arena") holds everything.
struct gfx_model {
  int hidden, layers, out_dim, feature_dim, edge_dim;
  int device;
  void *arena;
  float eps1[gfx::kMaxLayers];
  // fp32 tensors; index 0 = exact (GFX_F32 path), 1 = rounded to fp16 values
  // (what the GFX_F16 SIMT path multiplies by, so SIMT-F16 == UMMA-F16 inputs)
  const float *w_in[2];   // [H][F]
  const float *b_in;      // [H]
  const float *table[2];  // [L][edge_dim][H]
  const float *w1t[2];    // [L][H][2H]   (k-major rows: w1t[k][n] = W1'[n][k])
  const float *b1;        // [L][2H]
  const float *w2t[2];    // [L][2H][H]
  const float *b2;        // [L][H]
  const float *ln_g;      // [L][H]
  const float *ln_b;      // [L][H]
  const float *wat[2];    // [H][H]
  const float *ba;        // [H]
  const float *wbt[2];    // [H][O]
  const float *bb;        // [O]
  // fp16 images laid out exactly as the tcgen05 kernels want them in shared
  // memory (K-major, 128-byte swizzle, 64-column K blocks); see gfx_umma.cu
  const __half *w1_img;   // [L] x (2 kblocks x 256 rows x 64)   = 64 KB each
  const __half *w2_img;   // [L] x (4 kblocks x 128 rows x 64)   = 64 KB each
  const __half *wa_img;   //       (2 kblocks x 128 rows x 64)   = 32 KB
  const __half *wb_img;   //       (2 kblocks x 128 rows x 64)   = 32 KB
  const __half *table16;  // [L][edge_dim][H] fp16 (fused layer kernel)
  // lo parts of the same images, lo = fp16(w - fp16(w)): the split-fp16 tensor-core kernels of
  // the fp32 path (gfx_split9.cu) multiply by hi + lo
  const __half *w1_lo_img, *w2_lo_img, *wa_lo_img, *wb_lo_img;
  gfx_host_vectors host;
};
