// Sparse descriptor sampling and two-way nearest-neighbour matching (SURVEY 8f rank 3): the step after NMS in
// export_descriptor / evaluation.
// Reference (Gabriel-SGama/Semantic-SuperPoint):
//   models/model_wrap.py:295-313  SuperPointFrontend_torch.sample_desc_from_points
//        x_n = x / (W/2) - 1, y_n = y / (H/2) - 1 (float64, then .float());  F.grid_sample(coarse_desc, ., align_corners=True)
//        (bilinear, zero padding);  desc /= ||desc||_2 per point
//   models/model_wrap.py:451-494  PointTracker.nn_match_two_way
//        dmat = sqrt(2 - 2 clip(desc1^T desc2, -1, 1));  idx = argmin over axis 1, idx2 = argmin over axis 0;
//        keep = score < nn_thresh and idx2[idx] == arange
// The K1 x K2 distance matrix never reaches memory: each 64x64 tile reduces to per-row / per-column minima, merged
// with 64-bit atomicMin on (distance bits << 32 | index) keys -- ties resolve to the lowest index like np.argmin.
#include "common.cuh"

// ----------------------------------------------------------------------------------------------
// descriptor sampling: block (k, i) = keypoint k of image i, thread = channel (strided).  Image i samples its first
// n_i = min(counts[i], limit) points; its columns k >= n_i are written as zeros.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sample_desc_kernel(const float* __restrict__ coarse, const double* __restrict__ pts, int capacity,
                   const unsigned int* __restrict__ counts, int limit, int D, int Hc, int Wc, int cell,
                   float* __restrict__ desc) {
  __shared__ float red[32];
  const int k = blockIdx.x, img = blockIdx.y;
  const size_t plane = (size_t)Hc * Wc;
  coarse += (size_t)img * D * plane;
  pts += (size_t)img * 3 * capacity;
  desc += (size_t)img * D * limit;
  if (k >= (int)min(counts[img], (unsigned int)limit)) {
    for (int c = threadIdx.x; c < D; c += blockDim.x) desc[(size_t)c * limit + k] = 0.f;
    return;
  }
  const double Wd = (double)(Wc * cell), Hd = (double)(Hc * cell);
  // pts is the reference's [3,K] (x row, y row, conf row) float64 array, rows `capacity` apart
  const float xn = (float)(pts[k] / (Wd / 2.0) - 1.0);
  const float yn = (float)(pts[(size_t)capacity + k] / (Hd / 2.0) - 1.0);
  const float ix = ((xn + 1.f) / 2.f) * (float)(Wc - 1);
  const float iy = ((yn + 1.f) / 2.f) * (float)(Hc - 1);
  const float fx = floorf(ix), fy = floorf(iy);
  const bool any = fx >= -1.f && fx < (float)Wc && fy >= -1.f && fy < (float)Hc;
  const int x0 = any ? (int)fx : 0, y0 = any ? (int)fy : 0, x1 = x0 + 1, y1 = y0 + 1;
  const float wx1 = ix - fx, wx0 = (fx + 1.f) - ix, wy1 = iy - fy, wy0 = (fy + 1.f) - iy;
  const bool xin0 = any && x0 >= 0, xin1 = any && x1 < Wc, yin0 = any && y0 >= 0, yin1 = any && y1 < Hc;
  float ss = 0.f;
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    const float* p = coarse + (size_t)c * plane;
    float v = 0.f;  // accumulation order of torch's CPU grid_sample: nw, ne, sw, se
    if (yin0 && xin0) v += __ldg(p + (size_t)y0 * Wc + x0) * (wx0 * wy0);
    if (yin0 && xin1) v += __ldg(p + (size_t)y0 * Wc + x1) * (wx1 * wy0);
    if (yin1 && xin0) v += __ldg(p + (size_t)y1 * Wc + x0) * (wx0 * wy1);
    if (yin1 && xin1) v += __ldg(p + (size_t)y1 * Wc + x1) * (wx1 * wy1);
    desc[(size_t)c * limit + k] = v;
    ss = fmaf(v, v, ss);
  }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) tot += red[w];
  const float nrm = sqrtf(tot);
  for (int c = threadIdx.x; c < D; c += blockDim.x) {  // each thread rescales the values it wrote
    float* o = desc + (size_t)c * limit + k;
    *o = *o / nrm;  // 0/0 = NaN for a point sampled entirely outside, like the reference
  }
}

extern "C" int ssp_sample_desc_batch(const float* coarse, const double* pts, int capacity, const unsigned int* counts,
                                     int limit, int I, int D, int Hc, int Wc, int cell, float* desc, void* stream) {
  SSP_REQUIRE(coarse && pts && counts && desc, "ssp_sample_desc_batch: null pointer");
  SSP_REQUIRE(I > 0 && I <= 65535 && D > 0 && Hc > 0 && Wc > 0 && cell > 0 && limit > 0 && capacity >= limit,
              "ssp_sample_desc_batch: bad sizes I=%d D=%d Hc=%d Wc=%d limit=%d capacity=%d", I, D, Hc, Wc, limit, capacity);
  sample_desc_kernel<<<dim3(limit, I), 256, 0, (cudaStream_t)stream>>>(coarse, pts, capacity, counts, limit, D, Hc, Wc,
                                                                      cell, desc);
  SSP_CUDA_CHECK_LAUNCH("sample_desc_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// two-way nearest neighbour: 64x64 tiles of desc1^T desc2, 16 channels per shared-memory step, 4x4 outputs per thread
// ----------------------------------------------------------------------------------------------
#define NN_T 64
#define NN_KC 16

__device__ __forceinline__ unsigned long long nn_key(float dist, int idx) {
  return ((unsigned long long)__float_as_uint(dist) << 32) | (unsigned int)idx;  // dist >= 0: bit order = value order
}

__global__ void __launch_bounds__(256)
nn_match_kernel(const float* __restrict__ d1, const float* __restrict__ d2, int D, int K1, int K2,
                unsigned long long* __restrict__ best1, unsigned long long* __restrict__ best2) {
  __shared__ __align__(16) float s1[NN_KC][NN_T], s2[NN_KC][NN_T];
  __shared__ unsigned long long rbest[NN_T], cbest[NN_T];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int i0 = blockIdx.y * NN_T, j0 = blockIdx.x * NN_T;
  if (tid < NN_T) {
    rbest[tid] = ~0ull;
    cbest[tid] = ~0ull;
  }
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  for (int c0 = 0; c0 < D; c0 += NN_KC) {
    __syncthreads();
    for (int e = tid; e < NN_KC * NN_T; e += 256) {
      int c = e / NN_T, p = e % NN_T;
      bool cok = c0 + c < D;
      s1[c][p] = (cok && i0 + p < K1) ? __ldg(d1 + (size_t)(c0 + c) * K1 + i0 + p) : 0.f;
      s2[c][p] = (cok && j0 + p < K2) ? __ldg(d2 + (size_t)(c0 + c) * K2 + j0 + p) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < NN_KC; ++c) {
      const float4 a4 = *reinterpret_cast<const float4*>(&s1[c][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&s2[c][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(a[u], b[v], acc[u][v]);
    }
  }
  // distances, tile minima
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + ty * 4 + u;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int j = j0 + tx * 4 + v;
      if (i < K1 && j < K2) {
        float dot = fminf(fmaxf(acc[u][v], -1.f), 1.f);
        float dist = sqrtf(2.f - 2.f * dot);
        atomicMin(&rbest[ty * 4 + u], nn_key(dist, j));
        atomicMin(&cbest[tx * 4 + v], nn_key(dist, i));
      }
    }
  }
  __syncthreads();
  if (tid < NN_T) {
    if (i0 + tid < K1 && rbest[tid] != ~0ull) atomicMin(best1 + i0 + tid, rbest[tid]);
  } else if (tid < 2 * NN_T) {
    int t = tid - NN_T;
    if (j0 + t < K2 && cbest[t] != ~0ull) atomicMin(best2 + j0 + t, cbest[t]);
  }
}

// best1 [K1], best2 [K2]: (distance bits << 32 | index of the nearest descriptor of the other set); set to ~0 here.
extern "C" int ssp_nn_match(const float* desc1, const float* desc2, int D, int K1, int K2,
                            unsigned long long* best1, unsigned long long* best2, void* stream) {
  SSP_REQUIRE(desc1 && desc2 && best1 && best2, "ssp_nn_match: null pointer");
  SSP_REQUIRE(D > 0 && K1 > 0 && K2 > 0, "ssp_nn_match: bad sizes D=%d K1=%d K2=%d", D, K1, K2);
  cudaStream_t st = (cudaStream_t)stream;
  SSP_CUDA_CALL(cudaMemsetAsync(best1, 0xff, (size_t)K1 * 8, st));
  SSP_CUDA_CALL(cudaMemsetAsync(best2, 0xff, (size_t)K2 * 8, st));
  dim3 grid(ssp_ceil_div(K2, NN_T), ssp_ceil_div(K1, NN_T));
  nn_match_kernel<<<grid, 256, 0, st>>>(desc1, desc2, D, K1, K2, best1, best2);
  SSP_CUDA_CHECK_LAUNCH("nn_match_kernel");
  return SSP_OK;
}
