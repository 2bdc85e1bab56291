// Host-side TMA descriptors of the packed bf16 descriptor planes (ssp_desc_pack's [rows, 256] hi / lo layout), shared by
// the tcgen05 kernels of the descriptor loss (desc_tc.cu) and of the keypoint matcher (match_tc.cu).
#pragma once
#include "common.cuh"
#include <cuda.h>

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// hi (+ lo) planes [rows, 256] bf16 as ONE 3-D tensor {256 channels, rows, planes}: a [64 ch x box_rows x planes] box brings
// the same cells of both planes with one TMA instruction.  The planes may live anywhere as long as lo is above hi and the
// distance is a multiple of 16 bytes (the Python host allocates them back to back).
static inline int make_planes_map3(CUtensorMap* m, const void* hi, const void* lo, uint64_t rows, uint32_t box_rows) {
  constexpr uint64_t kChannels = 256;  // descriptor channels = GEMM K
  constexpr uint32_t kChunk = 64;      // channels per box = 128 B of bf16 = one swizzle row
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) { ssp_set_error("cuTensorMapEncodeTiled unavailable (driver too old?)"); return SSP_EUNSUPPORTED; }
  const uint64_t plane_bytes = rows * kChannels * 2;
  uint64_t pstride = plane_bytes;
  if (lo) {
    if ((uintptr_t)lo <= (uintptr_t)hi || (((uintptr_t)lo - (uintptr_t)hi) & 15) || ((uintptr_t)lo - (uintptr_t)hi) < plane_bytes ||
        ((uintptr_t)lo - (uintptr_t)hi) >= (1ull << 40)) {
      ssp_set_error("tcgen05 descriptor kernels: the lo plane must lie above the hi plane (distance a multiple of 16 bytes)");
      return SSP_EARG;
    }
    pstride = (uintptr_t)lo - (uintptr_t)hi;
  }
  cuuint64_t dims[3] = {(cuuint64_t)kChannels, (cuuint64_t)rows, (cuuint64_t)(lo ? 2 : 1)};
  cuuint64_t strides[2] = {(cuuint64_t)kChannels * 2, (cuuint64_t)pstride};
  cuuint32_t box[3] = {kChunk, box_rows, (cuuint32_t)(lo ? 2 : 1)};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(hi), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { ssp_set_error("cuTensorMapEncodeTiled (3-D planes) failed with CUresult %d", (int)r); return SSP_EARG; }
  return SSP_OK;
}
