// Shared helpers for the ssp_b200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#define SSP_OK 0
#define SSP_EARG -1       // bad argument (null pointer, non-positive size, misalignment)
#define SSP_EUNSUPPORTED -2

// thread-local last error text, read through ssp_last_error()
void ssp_set_error(const char* fmt, ...);

#define SSP_REQUIRE(cond, ...)            \
  do {                                    \
    if (!(cond)) {                        \
      ssp_set_error(__VA_ARGS__);         \
      return SSP_EARG;                    \
    }                                     \
  } while (0)

#define SSP_CUDA_CHECK_LAUNCH(name)                                                        \
  do {                                                                                     \
    cudaError_t e__ = cudaGetLastError();                                                  \
    if (e__ != cudaSuccess) {                                                              \
      ssp_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));               \
      return (int)e__;                                                                     \
    }                                                                                      \
  } while (0)

#define SSP_CUDA_CALL(expr)                                                                \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      ssp_set_error("%s failed: %s", #expr, cudaGetErrorString(e__));                      \
      return (int)e__;                                                                     \
    }                                                                                      \
  } while (0)

static inline int ssp_ceil_div(int a, int b) { return (a + b - 1) / b; }

// number of SMs of the current device (cached); 148 on B200
int ssp_num_sms();

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of doubles; result valid in thread 0. `sh` must hold >= 32 doubles.
__device__ __forceinline__ double block_sum_d(double v, double* sh) {
  v = warp_sum_d(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  double r = 0.0;
  if (w == 0) {
    r = lane < nw ? sh[lane] : 0.0;
    r = warp_sum_d(r);
  }
  return r;
}

// Homography applied to one point, same operation order everywhere in the library:
//   X = h0*x + h1*y + h2 (fma chain), then xy / z.   (reference: utils/utils.py:337-342)
__device__ __forceinline__ void homography_apply(const float* __restrict__ h, float x, float y,
                                                 float& ox, float& oy) {
  float X = fmaf(h[1], y, h[0] * x) + h[2];
  float Y = fmaf(h[4], y, h[3] * x) + h[5];
  float Z = fmaf(h[7], y, h[6] * x) + h[8];
  ox = X / Z;
  oy = Y / Z;
}

// float64 pixel-coordinate warp of the evaluation side, [x, y, 1] H^T / z (evaluations/detector_evaluation.py:139-150);
// warp_keypoints_f64_kernel and the evaluation kernels share it
__device__ __forceinline__ void warp_keypoint_f64(const double* __restrict__ Hm, double x, double y, double& ox, double& oy) {
  double X = Hm[0] * x + Hm[1] * y + Hm[2];
  double Y = Hm[3] * x + Hm[4] * y + Hm[5];
  double Z = Hm[6] * x + Hm[7] * y + Hm[8];
  ox = X / Z;
  oy = Y / Z;
}
