// Homography-adaptation heatmap aggregation.
// Reference: export.py:49-60 (combine_heatmap)  -- Gabriel-SGama/Semantic-SuperPoint
//   out = sum_n warp_n(heat_n * mask_n) / sum_n warp_n(mask_n), both warps bilinear with the same H_n.
// One kernel: the heat*mask product is formed at the gather, the N-sum stays in registers, the two
// intermediate [N,1,H,W] warped stacks of the reference never exist.  HBM traffic = the algorithmic
// (2N+1)*H*W*4 bytes.  A block owns an 8x8 output tile x 4 interleaved view groups.
#include "common.cuh"

#define CH_PIX 64
#define CH_GROUPS 4

// ncu of the first version (32 x 100 views of 240x320): 140 SASS instructions per (pixel, view), issue slots 63 % busy, DRAM 14 %:
// instruction-bound.  This version keeps the per-view work lean: homographies padded to 12 floats (three 16-byte shared loads),
// 32-bit tap offsets against per-view base pointers, the four corner predicates folded once.
// SIGNED = false: heat and a float mask, two gathers per tap (the reference's heat * mask product formed at the gather).
// SIGNED = true: heat is flatten_detection_masked's array (heat where the view's mask is 1, -1 where it is 0), so a tap is ONE
// gather and a sign test; mask is ignored and flag (its non-binary-mask flag, or NULL) turns the output into NaN.  The gather
// kernels are bound by L1 wavefronts (ncu: l1tex 89 %, ~6 lines per warp-wide load under rotation), so half the loads is what
// moves them.  Same arithmetic for m in {0, 1}: bit-identical results.
template <bool SIGNED>
__global__ void __launch_bounds__(CH_PIX * CH_GROUPS)
combine_heatmap_kernel(const float* __restrict__ heat, const float* __restrict__ mask,
                       const float* __restrict__ Hinv, int N, int H, int W, const float* __restrict__ xs,
                       const float* __restrict__ ys, const int* __restrict__ flag, float* __restrict__ out) {
  extern __shared__ __align__(16) float sh[];  // N x 12 floats (homography + pad), then 2*CH_PIX*CH_GROUPS partial sums
  float4* hs = reinterpret_cast<float4*>(sh);
  float* part = sh + N * 12;
  // blockIdx.y = source image (batched export: heat/mask [I,N,H,W], Hinv [I,N,3,3], out [I,H,W])
  const int plane = H * W;
  heat += (size_t)blockIdx.y * N * plane;
  mask += (size_t)blockIdx.y * N * plane;
  Hinv += (size_t)blockIdx.y * N * 9;
  out += (size_t)blockIdx.y * plane;
  for (int i = threadIdx.x; i < N * 12; i += blockDim.x) {
    const int n = i / 12, k = i - n * 12;
    sh[i] = k < 9 ? Hinv[n * 9 + k] : 0.f;
  }
  __syncthreads();
  const int lp = threadIdx.x % CH_PIX, g = threadIdx.x / CH_PIX;
  // a block owns an 8x8 pixel tile, a warp an 8x4 patch: under any rotation the bilinear footprints of a warp
  // stay inside a compact source patch (few 32 B sectors per gather instead of one per lane)
  const int tiles_x = (W + 7) / 8;
  const int x = (blockIdx.x % tiles_x) * 8 + (lp & 7), y = (blockIdx.x / tiles_x) * 8 + (lp >> 3);
  const bool inside = x < W && y < H;
  float sum_h = 0.f, sum_m = 0.f;
  if (inside) {
    const float gx = __ldg(xs + x), gy = __ldg(ys + y);
    const float fW = (float)W, fH = (float)H, sx = (float)(W - 1), sy = (float)(H - 1);
    const float* hp = heat + (size_t)g * plane;
    const float* mp = mask + (size_t)g * plane;
    const size_t step = (size_t)CH_GROUPS * plane;
    for (int n = g; n < N; n += CH_GROUPS, hp += step, mp += step) {
      const float4 h0 = hs[3 * n], h1 = hs[3 * n + 1], h2 = hs[3 * n + 2];  // h0..h3 | h4..h7 | h8
      // same operation order as homography_apply / grid_sampler_unnormalize (align_corners=True)
      const float X = fmaf(h0.y, gy, h0.x * gx) + h0.z;
      const float Y = fmaf(h1.x, gy, h0.w * gx) + h1.y;
      const float Z = fmaf(h1.w, gy, h1.z * gx) + h2.x;
      const float ix = ((X / Z + 1.f) / 2.f) * sx;
      const float iy = ((Y / Z + 1.f) / 2.f) * sy;
      const float fx = floorf(ix), fy = floorf(iy);
      // reject views whose 2x2 footprint is entirely outside (also keeps the int casts in range)
      if (!(fx >= -1.f && fx < fW && fy >= -1.f && fy < fH)) continue;
      const int x0 = (int)fx, y0 = (int)fy;
      const float wx1 = ix - fx, wx0 = (fx + 1.f) - ix;
      const float wy1 = iy - fy, wy0 = (fy + 1.f) - iy;
      const bool xin0 = x0 >= 0, xin1 = x0 + 1 < W, yin0 = y0 >= 0, yin1 = y0 + 1 < H;
      const int o = y0 * W + x0;
      float ah = 0.f, am = 0.f;
      if constexpr (SIGNED) {
        // out-of-image taps read as "masked"
        const float p00 = (yin0 && xin0) ? __ldg(hp + o) : -1.f;
        const float p01 = (yin0 && xin1) ? __ldg(hp + o + 1) : -1.f;
        const float p10 = (yin1 && xin0) ? __ldg(hp + o + W) : -1.f;
        const float p11 = (yin1 && xin1) ? __ldg(hp + o + W + 1) : -1.f;
        if (p00 >= 0.f) { const float w = wx0 * wy0; am += w; ah += p00 * w; }
        if (p01 >= 0.f) { const float w = wx1 * wy0; am += w; ah += p01 * w; }
        if (p10 >= 0.f) { const float w = wx0 * wy1; am += w; ah += p10 * w; }
        if (p11 >= 0.f) { const float w = wx1 * wy1; am += w; ah += p11 * w; }
      } else {
        if (yin0 && xin0) { const float m = __ldg(mp + o), w = wx0 * wy0; am += m * w; ah += (__ldg(hp + o) * m) * w; }
        if (yin0 && xin1) { const float m = __ldg(mp + o + 1), w = wx1 * wy0; am += m * w; ah += (__ldg(hp + o + 1) * m) * w; }
        if (yin1 && xin0) { const float m = __ldg(mp + o + W), w = wx0 * wy1; am += m * w; ah += (__ldg(hp + o + W) * m) * w; }
        if (yin1 && xin1) { const float m = __ldg(mp + o + W + 1), w = wx1 * wy1; am += m * w; ah += (__ldg(hp + o + W + 1) * m) * w; }
      }
      sum_h += ah;
      sum_m += am;
    }
  }
  part[threadIdx.x] = sum_h;
  part[CH_PIX * CH_GROUPS + threadIdx.x] = sum_m;
  __syncthreads();
  if (g == 0 && inside) {
    float th = 0.f, tm = 0.f;
#pragma unroll
    for (int q = 0; q < CH_GROUPS; ++q) {
      th += part[q * CH_PIX + lp];
      tm += part[CH_PIX * CH_GROUPS + q * CH_PIX + lp];
    }
    float r = th / tm;  // 0/0 -> NaN exactly like the reference when no view covers the pixel
    if constexpr (SIGNED) {
      if (flag && *flag) r = __int_as_float(0x7fc00000);  // a mask that was not 0/1: refuse loudly
    }
    out[y * W + x] = r;
  }
}

template <bool SIGNED>
static int combine_launch(const char* name, const float* heat, const float* mask, const float* Hinv, int I, int N, int H,
                          int W, const float* xs, const float* ys, const int* flag, float* out, void* stream) {
  SSP_REQUIRE(I > 0 && I <= 65535 && N > 0 && H > 0 && W > 0, "%s: bad sizes I=%d N=%d H=%d W=%d", name, I, N, H, W);
  size_t smem = ((size_t)N * 12 + 2 * CH_PIX * CH_GROUPS) * sizeof(float);
  SSP_REQUIRE(smem <= 48 * 1024, "%s: N=%d views exceed the shared-memory table (max ~900)", name, N);
  dim3 nblk(ssp_ceil_div(W, 8) * ssp_ceil_div(H, 8), I);
  combine_heatmap_kernel<SIGNED><<<nblk, CH_PIX * CH_GROUPS, smem, (cudaStream_t)stream>>>(heat, mask, Hinv, N, H, W, xs, ys,
                                                                                          flag, out);
  SSP_CUDA_CHECK_LAUNCH("combine_heatmap_kernel");
  return SSP_OK;
}

extern "C" int ssp_combine_heatmap(const float* heat, const float* mask, const float* Hinv, int I, int N, int H, int W,
                                   const float* xs, const float* ys, float* out, void* stream) {
  SSP_REQUIRE(heat && mask && Hinv && xs && ys && out, "ssp_combine_heatmap: null pointer");
  return combine_launch<false>("ssp_combine_heatmap", heat, mask, Hinv, I, N, H, W, xs, ys, nullptr, out, stream);
}

// heat = flatten_detection_masked output [I,N,H,W]; flag = its non-binary-mask flag (device int) or NULL
extern "C" int ssp_combine_heatmap_signed(const float* heat, const float* Hinv, int I, int N, int H, int W, const float* xs,
                                          const float* ys, const int* flag, float* out, void* stream) {
  SSP_REQUIRE(heat && Hinv && xs && ys && out, "ssp_combine_heatmap_signed: null pointer");
  return combine_launch<true>("ssp_combine_heatmap_signed", heat, nullptr, Hinv, I, N, H, W, xs, ys, flag, out, stream);
}
