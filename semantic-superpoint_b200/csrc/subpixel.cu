// Sub-pixel refinement of NMS keypoints: SuperPointFrontend_torch.soft_argmax_points (models/model_wrap.py:212-248) with
// extract_patch_from_points, norm_patches, do_log and soft_argmax_2d of utils/losses.py, the last one being torchgeometry
// 0.1.2 SpatialSoftArgmax2d(normalized_coordinates=False).  The shipped COCO export config turns it on between NMS and
// top-k (configs/magicpoint_coco_export.yaml:44-45, export.py:309-314) -- Gabriel-SGama/Semantic-SuperPoint.
//
// One warp per point.  A patch has at most 15 x 15 = 225 taps, 8 per lane in registers; every reduction is a per-lane
// sum in tap order followed by an xor butterfly, so all lanes hold the same value and a point's result does not depend
// on the launch.  fp32 with accurate logf / expf / division (the library builds without fast math), in the reference's
// operation order; the coordinate update is float64 like the reference's `pts` array.
#include "common.cuh"
#include <math.h>

#define SAP_MAX_PATCH 15
#define SAP_TAPS_PER_LANE ((SAP_MAX_PATCH * SAP_MAX_PATCH + 31) / 32)
#define SAP_WARPS 8

// torch.max propagates NaN; fmaxf would drop it
__device__ __forceinline__ float max_nan(float a, float b) { return (a > b || a != a) ? a : b; }

__device__ __forceinline__ float warp_max_nan(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max_nan(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(SAP_WARPS * 32)
soft_argmax_points_kernel(const float* __restrict__ heat, int H, int W, double* __restrict__ pts, int capacity,
                          const unsigned int* __restrict__ counts, int limit, int patch) {
  const int img = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.x * SAP_WARPS + (threadIdx.x >> 5);
  const unsigned int K = min(counts[img], (unsigned int)limit);  // limit <= capacity (host)
  if ((unsigned int)k >= K) return;  // whole warp
  heat += (size_t)img * H * W;
  pts += (size_t)img * 3 * capacity;
  const double px = pts[k], py = pts[capacity + k];
  const int half = patch / 2;
  // extract_patch_from_points: np.pad(heat, patch // 2) then [yi : yi + patch, xi : xi + patch], (xi, yi) = astype(int)
  const int x0 = (int)px - half, y0 = (int)py - half;
  const int n = patch * patch;
  float v[SAP_TAPS_PER_LANE];
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < SAP_TAPS_PER_LANE; ++j) {
    const int t = lane + 32 * j;
    const int r = t / patch, c = t - r * patch;
    const int y = y0 + r, x = x0 + c;
    v[j] = (t < n && y >= 0 && y < H && x >= 0 && x < W) ? heat[(size_t)y * W + x] : 0.f;
    sum += v[j];
  }
  // norm_patches: q = patch / (sum + 1e-6); do_log: q < 0 -> 1e-6, log (a zero tap gives -inf)
  const float d = warp_sum(sum) + 1e-6f;
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < SAP_TAPS_PER_LANE; ++j) {
    if (lane + 32 * j < n) {
      float q = v[j] / d;
      if (q < 0.f) q = 1e-6f;
      v[j] = logf(q);
      m = max_nan(m, v[j]);
    }
  }
  m = warp_max_nan(m);
  // SpatialSoftArgmax2d: e = exp(l - max l), s = 1 / (sum e + 1e-6), expected coordinate = sum((pos * e) * s)
  float es = 0.f;
#pragma unroll
  for (int j = 0; j < SAP_TAPS_PER_LANE; ++j) {
    v[j] = lane + 32 * j < n ? expf(v[j] - m) : 0.f;
    es += v[j];
  }
  const float s = 1.0f / (warp_sum(es) + 1e-6f);
  float sx = 0.f, sy = 0.f;
#pragma unroll
  for (int j = 0; j < SAP_TAPS_PER_LANE; ++j) {
    const int t = lane + 32 * j;
    if (t < n) {
      const int r = t / patch, c = t - r * patch;
      sx += ((float)c * v[j]) * s;
      sy += ((float)r * v[j]) * s;
    }
  }
  sx = warp_sum(sx);
  sy = warp_sum(sy);
  if (lane == 0) {  // points[:, :2] + dxdy - patch_size // 2, float64
    pts[k] = (px + (double)sx) - (double)half;
    pts[capacity + k] = (py + (double)sy) - (double)half;
  }
}

extern "C" int ssp_soft_argmax_points(const float* heat, int I, int H, int W, double* pts, int capacity,
                                      const unsigned int* counts, int limit, int patch, void* stream) {
  SSP_REQUIRE(heat && pts && counts, "ssp_soft_argmax_points: null pointer");
  SSP_REQUIRE(patch >= 1 && patch <= SAP_MAX_PATCH, "ssp_soft_argmax_points: patch must be in 1..%d, got %d", SAP_MAX_PATCH,
              patch);
  SSP_REQUIRE(I > 0 && I <= 65535 && H > 0 && W > 0 && capacity > 0 && limit >= 0,
              "ssp_soft_argmax_points: bad sizes I=%d H=%d W=%d capacity=%d limit=%d", I, H, W, capacity, limit);
  limit = limit < capacity ? limit : capacity;
  if (limit == 0) return SSP_OK;
  dim3 grid(ssp_ceil_div(limit, SAP_WARPS), I);
  soft_argmax_points_kernel<<<grid, SAP_WARPS * 32, 0, (cudaStream_t)stream>>>(heat, H, W, pts, capacity, counts, limit,
                                                                                 patch);
  SSP_CUDA_CHECK_LAUNCH("soft_argmax_points_kernel");
  return SSP_OK;
}
