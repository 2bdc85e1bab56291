// Batched homography warping: warp_points, inv_warp_image_batch, compute_valid_mask, filter masks.
// Reference semantics: utils/utils.py:303-405, 715-742 and evaluations/detector_evaluation.py:139-191
// (Gabriel-SGama/Semantic-SuperPoint).  All kernels are HBM-bound streaming kernels; the source
// image of a warp is gathered through L1/L2 (one image is 0.3-1.2 MB, far below the 126 MB L2).
#include "common.cuh"

// ----------------------------------------------------------------------------------------------
// a1 / a10: warp_points   out[b,p,:] = (H_b [x,y,1]^T)[:2] / (H_b [x,y,1]^T)[2]
// keep (optional) = the in-bounds predicate of filter_points: 0 <= p <= shape-1, inclusive.
// ----------------------------------------------------------------------------------------------
__global__ void warp_points_mask_kernel(const float* __restrict__ pts, int P, const float* __restrict__ Hm,
                                        float sx, float sy, float* __restrict__ out,
                                        uint8_t* __restrict__ keep) {
  int b = blockIdx.y;
  __shared__ float h[9];
  if (threadIdx.x < 9) h[threadIdx.x] = Hm[b * 9 + threadIdx.x];
  __syncthreads();
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
    float2 xy = reinterpret_cast<const float2*>(pts)[p];
    float ox, oy;
    homography_apply(h, xy.x, xy.y, ox, oy);
    reinterpret_cast<float2*>(out)[(size_t)b * P + p] = make_float2(ox, oy);
    if (keep) keep[(size_t)b * P + p] = (ox >= 0.f && ox <= sx - 1.f && oy >= 0.f && oy <= sy - 1.f) ? 1 : 0;
  }
}

extern "C" int ssp_warp_points_mask(const float* pts, int P, const float* Hm, int B, float shape_x,
                                    float shape_y, float* out, uint8_t* keep, void* stream) {
  SSP_REQUIRE(pts && Hm && out, "ssp_warp_points_mask: null pointer");
  SSP_REQUIRE(P >= 0 && B > 0, "ssp_warp_points_mask: bad sizes P=%d B=%d", P, B);
  if (P == 0) return SSP_OK;
  dim3 grid(min(ssp_ceil_div(P, 256), 148 * 8), B);
  warp_points_mask_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(pts, P, Hm, shape_x, shape_y, out, keep);
  SSP_CUDA_CHECK_LAUNCH("warp_points_mask_kernel");
  return SSP_OK;
}

// Evaluation-side twin in float64 pixel coordinates (detector_evaluation.py:139-191):
// warped = [x,y,1] H^T / z ; keep = 0 <= x < W and 0 <= y < H (strict upper bound).
__global__ void warp_keypoints_f64_kernel(const double* __restrict__ kp, int K, const double* __restrict__ Hm,
                                          double W, double Hh, double* __restrict__ out,
                                          uint8_t* __restrict__ keep) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K) return;
  double ox, oy;
  warp_keypoint_f64(Hm, kp[2 * i], kp[2 * i + 1], ox, oy);
  out[2 * i] = ox;
  out[2 * i + 1] = oy;
  keep[i] = (ox >= 0.0 && ox < W && oy >= 0.0 && oy < Hh) ? 1 : 0;
}

extern "C" int ssp_warp_keypoints_f64(const double* kp, int K, const double* Hm, double W, double H,
                                      double* out, uint8_t* keep, void* stream) {
  SSP_REQUIRE(kp && Hm && out && keep, "ssp_warp_keypoints_f64: null pointer");
  SSP_REQUIRE(K >= 0, "ssp_warp_keypoints_f64: bad K=%d", K);
  if (K == 0) return SSP_OK;
  warp_keypoints_f64_kernel<<<ssp_ceil_div(K, 128), 128, 0, (cudaStream_t)stream>>>(kp, K, Hm, W, H, out, keep);
  SSP_CUDA_CHECK_LAUNCH("warp_keypoints_f64_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// a2: inv_warp_image_batch = F.grid_sample(img, warp(grid), mode, zeros padding, align_corners=True)
// The normalised grid values xs[W], ys[H] are passed in as tables (the reference builds them with a
// CPU torch.linspace, utils/utils.py:375) so that sampling coordinates are reproduced exactly.
// ----------------------------------------------------------------------------------------------
// src pixel coordinate of output pixel (x,y): grid_sampler unnormalize with align_corners=True
__device__ __forceinline__ void src_coord(const float* h, float gx, float gy, int H, int W, float& ix, float& iy) {
  float nx, ny;
  homography_apply(h, gx, gy, nx, ny);
  ix = ((nx + 1.f) / 2.f) * (float)(W - 1);
  iy = ((ny + 1.f) / 2.f) * (float)(H - 1);
}

// Gather kernel.  One pixel per thread, 8x4-pixel warp patches (compact source footprint of a warp under rotation).
// The profile of the first version (ncu, 100 x 240 x 320) showed an INSTRUCTION-bound kernel (~190 SASS instructions per
// pixel, issue slots 65-85 % busy, DRAM 3 %): everything here is therefore about instruction count -- 32-bit index
// arithmetic against a per-image base pointer, bounds folded into four predicates, the homography in registers.
#define IWG_PX 4  // pixels per thread (rows y, y+8, y+16, y+24): 16 independent tap loads in flight per thread
template <int MODE>  // 0 bilinear, 1 nearest
__global__ void __launch_bounds__(256)
inv_warp_gather_kernel(const float* __restrict__ img, int C, int H, int W, const float* __restrict__ Hinv,
                       const float* __restrict__ xs, const float* __restrict__ ys, float* __restrict__ out) {
  const int b = blockIdx.z;
  const int tid = threadIdx.y * 32 + threadIdx.x, wrp = tid >> 5, lane = tid & 31;
  const int x = blockIdx.x * 32 + (wrp & 3) * 8 + (lane & 7);
  const int yb = blockIdx.y * (8 * IWG_PX) + (wrp >> 2) * 4 + (lane >> 3);
  if (x >= W) return;
  float h[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) h[i] = __ldg(Hinv + b * 9 + i);  // uniform address: one broadcast transaction each
  const float gx = __ldg(xs + x);
  const int plane = H * W;
  const float fW = (float)W, fH = (float)H;
  int off[IWG_PX][4];    // tap offsets, -1 = tap outside the image (contributes zero)
  float wgt[IWG_PX][4];
#pragma unroll
  for (int k = 0; k < IWG_PX; ++k) {
    const int y = yb + 8 * k;
#pragma unroll
    for (int t = 0; t < 4; ++t) { off[k][t] = -1; wgt[k][t] = 0.f; }
    if (y >= H) continue;
    float ix, iy;
    src_coord(h, gx, __ldg(ys + y), H, W, ix, iy);
    if (MODE == 0) {
      const float fx = floorf(ix), fy = floorf(iy);
      if (!(fx >= -1.f && fx < fW && fy >= -1.f && fy < fH)) continue;  // all four taps outside (keeps the int casts in range)
      const int x0 = (int)fx, y0 = (int)fy;
      const float wx1 = ix - fx, wx0 = (fx + 1.f) - ix, wy1 = iy - fy, wy0 = (fy + 1.f) - iy;
      const bool xin0 = x0 >= 0, xin1 = x0 + 1 < W, yin0 = y0 >= 0, yin1 = y0 + 1 < H;
      const int o = y0 * W + x0;
      // tap order and arithmetic of ATen's grid_sampler: nw, ne, sw, se
      if (yin0 && xin0) off[k][0] = o;
      if (yin0 && xin1) off[k][1] = o + 1;
      if (yin1 && xin0) off[k][2] = o + W;
      if (yin1 && xin1) off[k][3] = o + W + 1;
      wgt[k][0] = wx0 * wy0; wgt[k][1] = wx1 * wy0; wgt[k][2] = wx0 * wy1; wgt[k][3] = wx1 * wy1;
    } else {
      const float rx = rintf(ix), ry = rintf(iy);  // std::nearbyint under the default rounding mode = round half to even
      if (rx >= 0.f && rx < fW && ry >= 0.f && ry < fH) { off[k][0] = (int)ry * W + (int)rx; wgt[k][0] = 1.f; }
    }
  }
  const float* im = img + (size_t)b * C * plane;
  float* op = out + (size_t)b * C * plane + x;
  for (int c = 0; c < C; ++c, im += plane, op += plane) {
    float v[IWG_PX][4];
#pragma unroll
    for (int k = 0; k < IWG_PX; ++k)
#pragma unroll
      for (int t = 0; t < (MODE == 0 ? 4 : 1); ++t) v[k][t] = off[k][t] >= 0 ? __ldg(im + off[k][t]) : 0.f;
#pragma unroll
    for (int k = 0; k < IWG_PX; ++k) {
      const int y = yb + 8 * k;
      if (y >= H) continue;
      float acc;
      if (MODE == 0) {
        acc = 0.f;
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (off[k][t] >= 0) acc += v[k][t] * wgt[k][t];
      } else {
        acc = v[k][0];
      }
      op[y * W] = acc;
    }
  }
}

extern "C" int ssp_inv_warp_image(const float* img, int B, int C, int H, int W, const float* Hinv,
                                  const float* xs, const float* ys, int mode, float* out, void* stream) {
  SSP_REQUIRE(img && Hinv && xs && ys && out, "ssp_inv_warp_image: null pointer");
  SSP_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "ssp_inv_warp_image: bad sizes B=%d C=%d H=%d W=%d", B, C, H, W);
  SSP_REQUIRE(mode == 0 || mode == 1, "ssp_inv_warp_image: mode must be 0 (bilinear) or 1 (nearest); got %d", mode);
  SSP_REQUIRE(B <= 65535, "ssp_inv_warp_image: batch %d exceeds grid.z limit", B);
  dim3 block(32, 8);
  dim3 grid(ssp_ceil_div(W, 32), ssp_ceil_div(H, 8 * IWG_PX), B);
  if (mode == 0)
    inv_warp_gather_kernel<0><<<grid, block, 0, (cudaStream_t)stream>>>(img, C, H, W, Hinv, xs, ys, out);
  else
    inv_warp_gather_kernel<1><<<grid, block, 0, (cudaStream_t)stream>>>(img, C, H, W, Hinv, xs, ys, out);
  SSP_CUDA_CHECK_LAUNCH("inv_warp_gather_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// a3: compute_valid_mask = nearest-warp of an all-ones image, then cv2.erode with an explicit
// structuring element (taps that fall outside the image are ignored = cv2's default +inf border).
// Fused: a 32x32 output tile computes the raw in-bounds predicate for tile+halo into shared memory (bit packed)
// and takes the min over the kernel taps there; nothing but the final mask touches HBM.
// ----------------------------------------------------------------------------------------------
#define VM_TILE 32
// Rows of the tile + halo are packed into 64-bit words (bit = column) by warp ballots; the erosion of one output
// pixel is then kh shift / and / compare steps against the per-row masks of the structuring element instead of
// kh*kw byte reads.  Needs VM_TILE + kw - 1 <= 64, i.e. kw <= 33 (erosion radius <= 16).
__global__ void __launch_bounds__(256)
valid_mask_kernel(int H, int W, const float* __restrict__ Hinv, const float* __restrict__ xs,
                  const float* __restrict__ ys, const uint8_t* __restrict__ kern, int kh, int kw, int ax, int ay,
                  float* __restrict__ out) {
  __shared__ unsigned long long rowbits[VM_TILE + 64];  // one word per tile+halo row, 1 = valid or outside the image
  __shared__ unsigned long long kmask[64];              // structuring element rows
  __shared__ float h[9];
  const int b = blockIdx.z;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, lane = tid & 31, wrp = tid >> 5;
  if (tid < 9) h[tid] = Hinv[b * 9 + tid];
  if (tid < kh) {
    unsigned long long m = 0ull;
    for (int kx = 0; kx < kw; ++kx) m |= (unsigned long long)(kern[tid * kw + kx] != 0) << kx;
    kmask[tid] = m;
  }
  __syncthreads();
  const int ph = kh > 0 ? kh - 1 : 0, pw = kw > 0 ? kw - 1 : 0;
  const int th = VM_TILE + ph, tw = VM_TILE + pw;
  const int y0 = blockIdx.y * VM_TILE - (kh > 0 ? ay : 0);
  const int x0 = blockIdx.x * VM_TILE - (kw > 0 ? ax : 0);
  for (int r = wrp; r < th; r += 8) {
    const int yy = y0 + r;
    unsigned long long word = 0ull;
    for (int half = 0; half * 32 < tw; ++half) {
      const int c = half * 32 + lane, xx = x0 + c;
      bool v = true;  // outside the image (or beyond the halo): ignored by the erosion
      if (c < tw && yy >= 0 && yy < H && xx >= 0 && xx < W) {
        float ix, iy;
        src_coord(h, __ldg(xs + xx), __ldg(ys + yy), H, W, ix, iy);
        float rx = rintf(ix), ry = rintf(iy);
        v = (rx >= 0.f && rx < (float)W && ry >= 0.f && ry < (float)H);
      }
      word |= (unsigned long long)__ballot_sync(0xffffffffu, v) << (32 * half);
    }
    if (lane == 0) rowbits[r] = word;
  }
  __syncthreads();
  for (int i = tid; i < VM_TILE * VM_TILE; i += 256) {
    const int ly = i / VM_TILE, lx = i % VM_TILE;
    const int y = blockIdx.y * VM_TILE + ly, x = blockIdx.x * VM_TILE + lx;
    if (y >= H || x >= W) continue;
    bool m = true;
    if (kh > 0 && kw > 0) {
      for (int ky = 0; ky < kh; ++ky) {
        const unsigned long long km = kmask[ky];
        m = m && (((rowbits[ly + ky] >> lx) & km) == km);
      }
    } else {
      m = (rowbits[ly] >> lx) & 1ull;
    }
    out[((size_t)b * H + y) * W + x] = m ? 1.f : 0.f;
  }
}

// erosion_radius = 0 (homography-adaptation export, datasets/Coco.py:284-288 with the default margin): the mask is the
// in-bounds predicate itself.  Lean streaming kernel: one pixel per thread, coalesced rows, no tile / halo machinery (the
// general kernel above spends ~140 instructions per pixel on it).
__global__ void __launch_bounds__(256)
valid_mask_r0_kernel(int H, int W, const float* __restrict__ Hinv, const float* __restrict__ xs,
                     const float* __restrict__ ys, float* __restrict__ out) {
  const int b = blockIdx.z;
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
  if (x >= W || y >= H) return;
  float h[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) h[i] = __ldg(Hinv + b * 9 + i);
  float ix, iy;
  src_coord(h, __ldg(xs + x), __ldg(ys + y), H, W, ix, iy);
  const float rx = rintf(ix), ry = rintf(iy);
  const bool v = rx >= 0.f && rx < (float)W && ry >= 0.f && ry < (float)H;
  out[((size_t)b * H + y) * W + x] = v ? 1.f : 0.f;
}

extern "C" int ssp_valid_mask(int B, int H, int W, const float* Hinv, const float* xs, const float* ys,
                              const uint8_t* kern, int kh, int kw, int ax, int ay, float* out, void* stream) {
  SSP_REQUIRE(Hinv && xs && ys && out, "ssp_valid_mask: null pointer");
  SSP_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "ssp_valid_mask: bad sizes B=%d H=%d W=%d", B, H, W);
  SSP_REQUIRE((kh == 0 && kw == 0) || (kern && kh > 0 && kw > 0 && kh <= 33 && kw <= 33 && ax >= 0 && ax < kw &&
                                       ay >= 0 && ay < kh),
              "ssp_valid_mask: bad structuring element kh=%d kw=%d anchor=(%d,%d)", kh, kw, ax, ay);
  dim3 block(32, 8);
  if (kh == 0 && kw == 0) {
    dim3 grid0(ssp_ceil_div(W, 32), ssp_ceil_div(H, 8), B);
    valid_mask_r0_kernel<<<grid0, block, 0, (cudaStream_t)stream>>>(H, W, Hinv, xs, ys, out);
    SSP_CUDA_CHECK_LAUNCH("valid_mask_r0_kernel");
    return SSP_OK;
  }
  dim3 grid(ssp_ceil_div(W, VM_TILE), ssp_ceil_div(H, VM_TILE), B);
  valid_mask_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(H, W, Hinv, xs, ys, kern, kh, kw, ax, ay, out);
  SSP_CUDA_CHECK_LAUNCH("valid_mask_kernel");
  return SSP_OK;
}
