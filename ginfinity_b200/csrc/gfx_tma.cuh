// Host-side tensor-map construction for the 2-D tiled TMA loads/stores used
// by the tcgen05 kernels.  The driver entry point is looked up at run time so
// that libgfx.so needs no link-time dependency on libcuda.
#pragma once
#include <cuda.h>

#include "gfx_common.cuh"

namespace gfx {
namespace tma {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      ptr = nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}

// [rows, 128] fp16 row-major; box = 64 columns x `box_rows` rows with the
// 128-byte swizzle, i.e. one K-block of a K-major UMMA operand.  Rows outside
// the tensor are zero-filled on load and clipped on store.
inline int make_rows128_map(CUtensorMap *map, const void *base, int64_t rows, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(GFX_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[2] = {cuuint64_t(kHidden), cuuint64_t(rows)};
  const cuuint64_t strides[1] = {cuuint64_t(kHidden) * 2};
  const cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS)
    return fail(GFX_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(rc)));
  return GFX_OK;
}

// [rows, cols] fp16 row-major, cols a multiple of 64 (e.g. the [rows, 256] hi | lo image of
// the fp32 search): the same box and swizzle as make_rows128_map, any of the cols / 64 blocks.
inline int make_rows_map(CUtensorMap *map, const void *base, int64_t rows, int cols, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(GFX_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  const cuuint64_t strides[1] = {cuuint64_t(cols) * 2};
  const cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS)
    return fail(GFX_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(rc)));
  return GFX_OK;
}

}  // namespace tma
}  // namespace gfx
