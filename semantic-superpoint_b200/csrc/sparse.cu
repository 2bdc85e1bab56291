// Sparse descriptor loss (SURVEY 8f rank 2): the loss every shipped training config uses.
// Reference: utils/loss_functions/sparse_loss.py:65-284 (descriptor_loss_sparse, batch_descriptor_loss_sparse) with
//            utils/loss_functions/pixelwise_contrastive_loss.py:140-265 (match_loss / non_match_descriptor_loss, dist="cos").
//
// Per image the reference samples K = num_matching_attempts cell correspondences (a, b) through the homography and
// Kn = K * num_masked_non_matches_per_match random non-matches on the HOST (numpy / torch CPU RNG) -- the sampled index lists
// are inputs here (semantic-superpoint_b200/sparse.py reproduces the sampling call for call) -- and then evaluates
//   match_b    = 1/K  sum_k max(1 - <D[:,a_k], Dw[:,b_k]>, 0)
//   nonmatch_b = sum_k max(<D[:,a'_k], Dw[:,b'_k]> - 0.2, 0) / (#{k: term > 0} + 1)
//   loss_b     = lamda_d * match_b + nonmatch_b;      outputs = means over the batch of (loss, match, nonmatch).
// Kernels: NCHW -> cell-major transpose (a gathered descriptor becomes one contiguous 1 KB row instead of 256 words 4*Nc bytes
// apart), one warp per sampled pair for the dot products, a fixed-order per-image reduction, and for the backward a
// warp-per-pair scatter (fp32 atomics into cell-major gradient buffers) followed by the transpose back.
#include "common.cuh"
#include "philox.cuh"
#include <cub/block/block_radix_sort.cuh>

// [B, Dch, Nc] <-> [B, Nc, Dch] through a 32 x 32 shared tile (both directions coalesced)
__global__ void __launch_bounds__(256)
sparse_transpose_kernel(const float* __restrict__ src, int rows, int cols, float* __restrict__ dst) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  src += (size_t)b * rows * cols;
  dst += (size_t)b * rows * cols;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = r0 + ty + 8 * k, c = c0 + tx;
    tile[ty + 8 * k][tx] = (r < rows && c < cols) ? __ldg(src + (size_t)r * cols + c) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c0 + ty + 8 * k, r = r0 + tx;
    if (r < rows && c < cols) dst[(size_t)c * rows + r] = tile[tx][ty + 8 * k];
  }
}

extern "C" int ssp_transpose_batched(const float* src, int B, int rows, int cols, float* dst, void* stream) {
  SSP_REQUIRE(src && dst, "ssp_transpose_batched: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && rows > 0 && cols > 0, "ssp_transpose_batched: bad sizes");
  dim3 grid(ssp_ceil_div(cols, 32), ssp_ceil_div(rows, 32), B);
  SSP_REQUIRE(grid.y <= 65535, "ssp_transpose_batched: too many rows");
  sparse_transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, rows, cols, dst);
  SSP_CUDA_CHECK_LAUNCH("sparse_transpose_kernel");
  return SSP_OK;
}

// dots[b, k] = <Dt[b, ia[b,k], :], Dwt[b, ib[b,k], :]>   (cell-major descriptors [B, Nc, Dch]); one warp per pair
__global__ void __launch_bounds__(256)
sparse_dots_kernel(const float* __restrict__ Dt, const float* __restrict__ Dwt, const int* __restrict__ ia,
                   const int* __restrict__ ib, int Kt, int Nc, int Dch, float* __restrict__ dots) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (k >= Kt) return;
  const int a = ia[(size_t)b * Kt + k], c = ib[(size_t)b * Kt + k];
  float acc = 0.f;
  if (a >= 0 && a < Nc && c >= 0 && c < Nc) {
    const float* pa = Dt + ((size_t)b * Nc + a) * Dch;
    const float* pc = Dwt + ((size_t)b * Nc + c) * Dch;
    for (int d = lane; d < Dch; d += 32) acc = fmaf(__ldg(pa + d), __ldg(pc + d), acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) dots[(size_t)b * Kt + k] = acc;
}

// per image, fixed summation order: stats[b] = { match_b, nonmatch_b, loss_b, hard count }
__global__ void __launch_bounds__(256)
sparse_reduce_kernel(const float* __restrict__ dots, int K, int Kn, float lamda, float mpos, float mneg,
                     float* __restrict__ stats) {
  __shared__ double shd[32];
  const int b = blockIdx.x;
  const float* dm = dots + (size_t)b * (K + Kn);
  const float* dn = dm + K;
  double sm = 0.0, sn = 0.0, hc = 0.0;
  for (int k = threadIdx.x; k < K; k += blockDim.x) sm += (double)fmaxf(mpos - dm[k], 0.f);
  for (int k = threadIdx.x; k < Kn; k += blockDim.x) {
    const float t = fmaxf(dn[k] - mneg, 0.f);
    sn += (double)t;
    hc += t != 0.f ? 1.0 : 0.0;  // torch.nonzero(non_match_loss): hard negatives
  }
  sm = block_sum_d(sm, shd);
  sn = block_sum_d(sn, shd);
  hc = block_sum_d(hc, shd);
  if (threadIdx.x == 0) {
    const float match = (float)(sm / (double)K);                    // 1/num_matches * sum
    const float nonmatch = (float)sn / ((float)hc + 1.f);           // sum / (num_hard_negatives + 1)
    stats[4 * b] = match;
    stats[4 * b + 1] = nonmatch;
    stats[4 * b + 2] = lamda * match + nonmatch;
    stats[4 * b + 3] = (float)hc;
  }
}

// batch means: out3 = { mean loss, mean match, mean nonmatch }   (torch.stack(...).mean(), sparse_loss.py:283-284)
__global__ void sparse_mean_kernel(const float* __restrict__ stats, int B, float* __restrict__ out3) {
  if (threadIdx.x == 0) {
    float l = 0.f, m = 0.f, n = 0.f;
    for (int b = 0; b < B; ++b) { m += stats[4 * b]; n += stats[4 * b + 1]; l += stats[4 * b + 2]; }
    out3[0] = l / (float)B;
    out3[1] = m / (float)B;
    out3[2] = n / (float)B;
  }
}

// Dt / Dwt: cell-major descriptors (ssp_transpose_batched of the NCHW tensors); ia / ib [B, K + Kn]: the K matches followed by the
// Kn non-matches (cell indices a in `descriptors`, b in `descriptors_warped`); dots [B, K + Kn] and stats [B, 4] are kept for
// the backward; out3 = the three returned scalars.
extern "C" int ssp_sparse_desc_loss_fwd(const float* Dt, const float* Dwt, const int* ia, const int* ib, int B, int Nc, int Dch,
                                        int K, int Kn, float lamda, float mpos, float mneg, float* dots, float* stats,
                                        float* out3, void* stream) {
  SSP_REQUIRE(Dt && Dwt && ia && ib && dots && stats && out3, "ssp_sparse_desc_loss_fwd: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Nc > 0 && Dch > 0 && K > 0 && Kn >= 0, "ssp_sparse_desc_loss_fwd: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  const int Kt = K + Kn;
  dim3 grid(ssp_ceil_div(Kt, 8), B);
  sparse_dots_kernel<<<grid, 256, 0, st>>>(Dt, Dwt, ia, ib, Kt, Nc, Dch, dots);
  SSP_CUDA_CHECK_LAUNCH("sparse_dots_kernel");
  sparse_reduce_kernel<<<B, 256, 0, st>>>(dots, K, Kn, lamda, mpos, mneg, stats);
  SSP_CUDA_CHECK_LAUNCH("sparse_reduce_kernel");
  sparse_mean_kernel<<<1, 32, 0, st>>>(stats, B, out3);
  SSP_CUDA_CHECK_LAUNCH("sparse_mean_kernel");
  return SSP_OK;
}

// backward: coefficient of every sampled pair, scattered into the cell-major gradients
//   match k:     -1/K * [mpos - dot >= 0] * (g_loss * lamda + g_match) / B        (torch.clamp passes the gradient at the bound)
//   non-match k:  1/(hard_b + 1) * [dot - mneg >= 0] * (g_loss + g_nonmatch) / B
//   dDt[b, a, :] += coef * Dwt[b, c, :],   dDwt[b, c, :] += coef * Dt[b, a, :]
__global__ void __launch_bounds__(256)
sparse_bwd_kernel(const float* __restrict__ Dt, const float* __restrict__ Dwt, const int* __restrict__ ia,
                  const int* __restrict__ ib, const float* __restrict__ dots, const float* __restrict__ stats,
                  const float* __restrict__ g3, int B, int Nc, int Dch, int K, int Kn, float lamda, float mpos, float mneg,
                  float* __restrict__ dDt, float* __restrict__ dDwt) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int Kt = K + Kn;
  const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (k >= Kt) return;
  const float dot = dots[(size_t)b * Kt + k];
  float coef;
  if (k < K) coef = (mpos - dot >= 0.f) ? -(g3[0] * lamda + g3[1]) / ((float)K * (float)B) : 0.f;
  else       coef = (dot - mneg >= 0.f) ? (g3[0] + g3[2]) / ((stats[4 * b + 3] + 1.f) * (float)B) : 0.f;
  if (coef == 0.f) return;
  const int a = ia[(size_t)b * Kt + k], c = ib[(size_t)b * Kt + k];
  if (a < 0 || a >= Nc || c < 0 || c >= Nc) return;
  const float* pa = Dt + ((size_t)b * Nc + a) * Dch;
  const float* pc = Dwt + ((size_t)b * Nc + c) * Dch;
  float* ga = dDt + ((size_t)b * Nc + a) * Dch;
  float* gc = dDwt + ((size_t)b * Nc + c) * Dch;
  for (int d = lane; d < Dch; d += 32) {
    atomicAdd(ga + d, coef * __ldg(pc + d));
    atomicAdd(gc + d, coef * __ldg(pa + d));
  }
}

// dDt / dDwt [B, Nc, Dch] are zeroed here; g3 = device { dL/dloss, dL/dmatch, dL/dnonmatch }
extern "C" int ssp_sparse_desc_loss_bwd(const float* Dt, const float* Dwt, const int* ia, const int* ib, const float* dots,
                                        const float* stats, const float* g3, int B, int Nc, int Dch, int K, int Kn,
                                        float lamda, float mpos, float mneg, float* dDt, float* dDwt, void* stream) {
  SSP_REQUIRE(Dt && Dwt && ia && ib && dots && stats && g3 && dDt && dDwt, "ssp_sparse_desc_loss_bwd: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Nc > 0 && Dch > 0 && K > 0 && Kn >= 0, "ssp_sparse_desc_loss_bwd: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)B * Nc * Dch * sizeof(float);
  SSP_CUDA_CALL(cudaMemsetAsync(dDt, 0, n, st));
  SSP_CUDA_CALL(cudaMemsetAsync(dDwt, 0, n, st));
  dim3 grid(ssp_ceil_div(K + Kn, 8), B);
  sparse_bwd_kernel<<<grid, 256, 0, st>>>(Dt, Dwt, ia, ib, dots, stats, g3, B, Nc, Dch, K, Kn, lamda, mpos, mneg, dDt, dDwt);
  SSP_CUDA_CHECK_LAUNCH("sparse_bwd_kernel");
  return SSP_OK;
}

// ------------------------------------------------------------------------------------------------------------------------
// Correspondence sampling on the device: the distribution of sample_correspondences (sparse_loss.py:170-255 with
// correspondence_finder.py:191-320), not its host RNG stream.  One block per image:
//   candidates  every cell a = (u, v) warped by T^-1 H T (scale_homography_torch, shift -1), rounded half to even, kept when
//               0 <= p <= (Wc-1, Hc-1); M = their count
//   matches     every candidate gets a 31-bit Philox key (non-candidates sort behind them) and one BlockRadixSort orders the
//               block: the first min(M, K) ranks are a uniformly random K-subset in random order (M >= K), or all M in random
//               order (M < K) followed by K - M draws with replacement from them -- crop_or_pad_choice (sparse_loss.py:44-48)
//   non-matches non_a[k n + j] = matches_a[k], non_b a uniform cell (the reference's perturbation is identically zero)
// Random numbers: Philox4x32-10, key = seed, counter = (item, image << 2 | purpose, launch counter).  The seed and the launch
// counter live in the caller's state buffer; every block reads the counter, and the last block to finish advances it, so
// consecutive launches (and graph replays) draw fresh lists with no host involvement.
// The purpose tags here (the low two bits of the counter's second word) are 0, 1 and 2; 3 belongs to homography.cu.
constexpr int SAMPLE_THREADS = 1024, SAMPLE_ITEMS = 8, SAMPLE_MAX_CELLS = SAMPLE_THREADS * SAMPLE_ITEMS;

__global__ void __launch_bounds__(SAMPLE_THREADS, 1)
sparse_sample_kernel(const float* __restrict__ mat_H, int Hc, int Wc, int K, int nper, unsigned long long* state, int* ia,
                     int* ib, int* Mout) {
  using Sort = cub::BlockRadixSort<unsigned, SAMPLE_THREADS, SAMPLE_ITEMS, int>;
  __shared__ typename Sort::TempStorage sort_tmp;
  __shared__ float hcell[9];
  __shared__ unsigned long long s_seed, s_ctr;
  __shared__ int s_count;
  const int b = blockIdx.x, t = threadIdx.x, Nc = Hc * Wc;
  const int Kn = K * nper, Kt = K + Kn;
  ia += (size_t)b * Kt;
  ib += (size_t)b * Kt;
  if (t == 0) {
    s_seed = *(volatile unsigned long long*)&state[0];
    s_ctr = *(volatile unsigned long long*)&state[1];
    s_count = 0;
    // T^-1 H T, T = [[2/Wc, 0, -1], [0, 2/Hc, -1], [0, 0, 1]] (sparse.py:20-24), in double and rounded once to fp32
    const float* h = mat_H + (size_t)b * 9;
    const double sx = 2.0 / Wc, sy = 2.0 / Hc;
    double ht[9];  // H T
    for (int r = 0; r < 3; ++r) {
      ht[3 * r] = (double)h[3 * r] * sx;
      ht[3 * r + 1] = (double)h[3 * r + 1] * sy;
      ht[3 * r + 2] = -(double)h[3 * r] - (double)h[3 * r + 1] + (double)h[3 * r + 2];
    }
    for (int c = 0; c < 3; ++c) {  // T^-1 = [[Wc/2, 0, Wc/2], [0, Hc/2, Hc/2], [0, 0, 1]]
      hcell[c] = (float)(0.5 * Wc * (ht[c] + ht[6 + c]));
      hcell[3 + c] = (float)(0.5 * Hc * (ht[3 + c] + ht[6 + c]));
      hcell[6 + c] = (float)ht[6 + c];
    }
  }
  __syncthreads();
  const uint2 key = make_uint2((unsigned)s_seed, (unsigned)(s_seed >> 32));
  const unsigned clo = (unsigned)s_ctr, chi = (unsigned)(s_ctr >> 32);

  // candidates, blocked arrangement: thread t holds cells 8t .. 8t+7
  unsigned keys[SAMPLE_ITEMS];
  int vals[SAMPLE_ITEMS];
  int mine = 0;
#pragma unroll
  for (int j = 0; j < SAMPLE_ITEMS; j += 4) {
    const uint4 r = philox4x32_10(make_uint4(t * (SAMPLE_ITEMS / 4) + j / 4, (unsigned)b << 2, clo, chi), key);
    const unsigned rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int cell = t * SAMPLE_ITEMS + j + q;
      keys[j + q] = 0xFFFFFFFFu;
      vals[j + q] = 0;
      if (cell < Nc) {
        const int v = cell / Wc, u = cell - v * Wc;
        float x, y;
        homography_apply(hcell, (float)u, (float)v, x, y);
        x = rintf(x);  // torch.round: half to even
        y = rintf(y);
        if (x >= 0.f && x <= (float)(Wc - 1) && y >= 0.f && y <= (float)(Hc - 1)) {
          keys[j + q] = rr[q] >> 1;
          vals[j + q] = cell | (((int)y * Wc + (int)x) << 16);
          ++mine;
        }
      }
    }
  }
  if (mine) atomicAdd(&s_count, mine);
  __syncthreads();
  const int M = s_count;
  Sort(sort_tmp).Sort(keys, vals);

  if (M == 0) {  // the homography maps no cell into the image: out-of-range lists (they contribute nothing), M[b] = 0 and the flag
    for (int k = t; k < Kt; k += SAMPLE_THREADS) {
      ia[k] = -1;
      ib[k] = -1;
    }
    if (t == 0) atomicAdd(&state[3], 1ull);
  } else {
#pragma unroll
    for (int j = 0; j < SAMPLE_ITEMS; ++j) {
      const int rank = t * SAMPLE_ITEMS + j;
      if (rank < M && rank < K) {
        ia[rank] = vals[j] & 0xFFFF;
        ib[rank] = vals[j] >> 16;
      }
    }
    __syncthreads();  // the block's global writes above are visible to the block from here on
    for (int k = M + t; k < K; k += SAMPLE_THREADS) {  // M < K: pad with draws with replacement from the M candidates
      const uint4 r = philox4x32_10(make_uint4(k, ((unsigned)b << 2) | 1u, clo, chi), key);
      const int src = uniform_below(r.x, r.y, M);
      ia[k] = ia[src];
      ib[k] = ib[src];
    }
    __syncthreads();
    for (int k = t; k < Kn; k += SAMPLE_THREADS) {
      const uint4 r = philox4x32_10(make_uint4(k, ((unsigned)b << 2) | 2u, clo, chi), key);
      ia[K + k] = ia[k / nper];
      ib[K + k] = uniform_below(r.x, r.y, Nc);
    }
  }
  if (t == 0) {
    Mout[b] = M;
    // the last block to finish advances the launch counter: every other block has read it by then
    __threadfence();
    const unsigned prev = atomicInc((unsigned*)&state[2], gridDim.x - 1);  // wraps back to 0 for the next launch
    if (prev == gridDim.x - 1) state[1] = s_ctr + 1;
  }
}

extern "C" int ssp_sparse_sample(const float* mat_H, int B, int Hc, int Wc, int K, int nper, unsigned long long* state, int* ia,
                                 int* ib, int* M, void* stream) {
  SSP_REQUIRE(mat_H && state && ia && ib && M, "ssp_sparse_sample: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Hc > 0 && Wc > 0, "ssp_sparse_sample: bad sizes");
  SSP_REQUIRE((long long)Hc * Wc <= SAMPLE_MAX_CELLS, "ssp_sparse_sample: %d x %d cells exceed the supported %d cells", Hc, Wc,
              SAMPLE_MAX_CELLS);
  SSP_REQUIRE(K > 0 && nper >= 0 && (long long)K * (nper + 1) <= 0x7FFFFFFF,
              "ssp_sparse_sample: need K > 0 and n >= 0 (got K = %d, n = %d)", K, nper);
  sparse_sample_kernel<<<B, SAMPLE_THREADS, 0, (cudaStream_t)stream>>>(mat_H, Hc, Wc, K, nper, state, ia, ib, M);
  SSP_CUDA_CHECK_LAUNCH("sparse_sample_kernel");
  return SSP_OK;
}

// out3 (ssp_sparse_desc_loss_fwd's batch means) becomes NaN when an image had no candidate (M[b] = 0); with total set,
// total = (det0[0] + det1[0]) + lambda_loss * out3[0], the sparse loss step's weighted sum (Train_model_heatmap_all.py:361-365)
__global__ void sparse_finalize_kernel(const int* __restrict__ M, int B, float* __restrict__ out3, const float* __restrict__ det0,
                                       const float* __restrict__ det1, float lambda_loss, float* __restrict__ total) {
  bool empty = false;
  if (M != nullptr)
    for (int b = threadIdx.x; b < B; b += 32) empty |= M[b] == 0;
  empty = __any_sync(0xffffffffu, empty);
  if (threadIdx.x == 0) {
    if (empty) out3[0] = out3[1] = out3[2] = __int_as_float(0x7fc00000);
    if (total != nullptr) total[0] = __fadd_rn(__fadd_rn(det0[0], det1[0]), __fmul_rn(lambda_loss, out3[0]));
  }
}

extern "C" int ssp_sparse_finalize(const int* M, int B, float* out3, const float* det0, const float* det1, float lambda_loss,
                                   float* total, void* stream) {
  SSP_REQUIRE(out3 && (total == nullptr || (det0 && det1)), "ssp_sparse_finalize: null pointer");
  SSP_REQUIRE(B > 0, "ssp_sparse_finalize: bad sizes");
  sparse_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(M, B, out3, det0, det1, lambda_loss, total);
  SSP_CUDA_CHECK_LAUNCH("sparse_finalize_kernel");
  return SSP_OK;
}
