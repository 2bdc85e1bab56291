// fp32 CUDA-core engine for the dense descriptor loss: exact-fp32 reference engine on the GPU
// (mode "fp32") and the cross-check for the tcgen05 engine.  Same outputs as desc_tc.cu:
// per-CTA partial sums of the negative hinge + the indicator bit-matrices, and the indicator GEMM of
// the backward.  Reference: utils/utils.py:863-890.
#include "desc_common.cuh"

#define ST 64   // tile edge
#define SK 16   // k chunk

__global__ void __launch_bounds__(256)
desc_dense_fwd_simt_kernel(const float* __restrict__ D, const float* __restrict__ Dw,
                           const float* __restrict__ mv_pad, DescGeom g,
                           double* __restrict__ partials, uint32_t* __restrict__ bitsR,
                           uint32_t* __restrict__ bitsC, float* __restrict__ dbgS) {
  __shared__ float As[SK][ST];
  __shared__ float Bs[SK][ST];
  __shared__ uint8_t pred[ST][ST + 4];
  __shared__ double shd[32];
  int b = blockIdx.z, r0 = blockIdx.y * ST, c0 = blockIdx.x * ST;
  int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const float* Db = D + (size_t)b * g.Dch * g.Nc;
  const float* Dwb = Dw + (size_t)b * g.Dch * g.Nc;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < g.Dch; k0 += SK) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int e = tid + 256 * q;
      int kk = e / ST, cc = e % ST;
      int k = k0 + kk;
      As[kk][cc] = (k < g.Dch && r0 + cc < g.Nc) ? __ldg(Db + (size_t)k * g.Nc + r0 + cc) : 0.f;
      Bs[kk][cc] = (k < g.Dch && c0 + cc < g.Nc) ? __ldg(Dwb + (size_t)k * g.Nc + c0 + cc) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SK; ++kk) {
      float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 bb = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  // fused epilogue
  float su = 0.f, sw = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int r = r0 + ty * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = c0 + tx * 4 + j;
      // zero padding gives dot = 0 -> hinge 0 (mneg > 0), so padded rows / columns need no masking
      float neg = fmaxf(acc[i][j] - g.mneg, 0.f);
      if (dbgS && r < g.Nc && c < g.Nc) dbgS[((size_t)b * g.Nc + r) * g.Nc + c] = acc[i][j];
      su += neg;
      sw = fmaf(neg, mv_pad[(size_t)b * g.Nc_pad + c], sw);
      pred[ty * 4 + i][tx * 4 + j] = neg > 0.f ? 1 : 0;
    }
  }
  double du = block_sum_d((double)su, shd);
  double dw = block_sum_d((double)sw, shd);
  if (tid == 0) {
    size_t cta = ((size_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    partials[2 * cta] = du;
    partials[2 * cta + 1] = dw;
  }
  if (bitsR) {
    __syncthreads();
    int NW = g.Nc_pad / 32;
    int q = tid % 64, wsel = (tid / 64) & 1;
    uint32_t word = 0;
    if (tid < 128) {
#pragma unroll 8
      for (int j = 0; j < 32; ++j) word |= (uint32_t)pred[q][wsel * 32 + j] << DESC_BITPOS(j);
      bitsR[((size_t)b * NW + c0 / 32 + wsel) * g.Nc_pad + r0 + q] = word;
    } else {
#pragma unroll 8
      for (int j = 0; j < 32; ++j) word |= (uint32_t)pred[wsel * 32 + j][q] << DESC_BITPOS(j);
      bitsC[((size_t)b * NW + r0 / 32 + wsel) * g.Nc_pad + c0 + q] = word;
    }
  }
}

extern "C" int ssp_desc_dense_simt_nblocks(int B, int Nc) {
  int t = desc_nc_pad(Nc) / ST;
  return B * t * t;
}

extern "C" int ssp_desc_dense_fwd_simt(const float* D, const float* Dw, const float* mv_pad, int B, int Hc, int Wc,
                                       int Dch, float mneg, double* partials, uint32_t* bitsR, uint32_t* bitsC,
                                       float* dbgS, void* stream) {
  SSP_REQUIRE(D && Dw && mv_pad && partials, "ssp_desc_dense_fwd_simt: null pointer");
  SSP_REQUIRE(mneg > 0.f, "ssp_desc_dense_fwd_simt: margin_neg must be > 0 (zero padding relies on it)");
  SSP_REQUIRE((bitsR == nullptr) == (bitsC == nullptr), "ssp_desc_dense_fwd_simt: bitsR/bitsC must both be given or both null");
  DescGeom g;
  g.B = B; g.Hc = Hc; g.Wc = Wc; g.Nc = Hc * Wc; g.Nc_pad = desc_nc_pad(g.Nc); g.Dch = Dch; g.cell = 0;
  g.dist = 0.f; g.lamda = 0.f; g.mpos = 0.f; g.mneg = mneg;
  SSP_REQUIRE(B > 0 && B <= 65535 && Hc > 0 && Wc > 0 && Dch > 0, "ssp_desc_dense_fwd_simt: bad sizes");
  int t = g.Nc_pad / ST;
  dim3 grid(t, t, B);
  desc_dense_fwd_simt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      D, Dw, mv_pad, g, partials, bitsR, bitsC, dbgS);
  SSP_CUDA_CHECK_LAUNCH("desc_dense_fwd_simt_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// indicator GEMM (backward):  out[b, d, r] = rowscale[b,r] * sum_k bit(r, k) * colscale[b,k] * src[b, d, k]
//   bits[b, kw, r] holds bits k = 32kw..32kw+31 of row r (element j at bit DESC_BITPOS(j)).  CTA = 32 rows r x 256 channels d.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
desc_bits_gemm_simt_kernel(const uint32_t* __restrict__ bits, const float* __restrict__ src,
                           const float* __restrict__ colscale, const float* __restrict__ rowscale, int Dch, int Nc,
                           int Nc_pad, float* __restrict__ out) {
  __shared__ float sv[256][33];
  __shared__ uint32_t wb[32];
  int b = blockIdx.y, r0 = blockIdx.x * 32, d0 = blockIdx.z * 256;
  int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  int NW = Nc_pad / 32;
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  for (int kw = 0; kw < NW; ++kw) {
    int k = kw * 32 + lane;
    if (kw * 32 >= Nc) break;
    __syncthreads();
    if (w == 0) wb[lane] = bits[((size_t)b * NW + kw) * Nc_pad + r0 + lane];
    float cs = 0.f;
    if (k < Nc) cs = colscale ? colscale[(size_t)b * Nc_pad + k] : 1.f;
    for (int dd = w; dd < 256; dd += 8) {
      int d = d0 + dd;
      sv[dd][lane] = (d < Dch && k < Nc) ? __ldg(src + ((size_t)b * Dch + d) * Nc + k) * cs : 0.f;
    }
    __syncthreads();
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = sv[tid][j];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      uint32_t word = wb[i];
      if (word == 0u) continue;
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (word & (1u << DESC_BITPOS(j))) acc[i] += v[j];
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; ++i) sv[tid][i] = acc[i];
  __syncthreads();
  int r = r0 + lane;
  if (r < Nc) {
    float rs = rowscale ? rowscale[(size_t)b * Nc_pad + r] : 1.f;
    for (int dd = w; dd < 256; dd += 8) {
      int d = d0 + dd;
      if (d < Dch) out[((size_t)b * Dch + d) * Nc + r] = sv[dd][lane] * rs;
    }
  }
}

extern "C" int ssp_desc_bits_gemm_simt(const uint32_t* bits, const float* src, const float* colscale,
                                       const float* rowscale, int B, int Dch, int Nc, float* out, void* stream) {
  SSP_REQUIRE(bits && src && out, "ssp_desc_bits_gemm_simt: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Dch > 0 && Nc > 0, "ssp_desc_bits_gemm_simt: bad sizes");
  int Nc_pad = desc_nc_pad(Nc);
  dim3 grid(Nc_pad / 32, B, ssp_ceil_div(Dch, 256));
  desc_bits_gemm_simt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(bits, src, colscale, rowscale, Dch, Nc, Nc_pad, out);
  SSP_CUDA_CHECK_LAUNCH("desc_bits_gemm_simt_kernel");
  return SSP_OK;
}
