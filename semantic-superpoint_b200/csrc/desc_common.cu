// Descriptor-loss kernels shared by both GEMM engines: geometry, exact positive pairs (fwd/bwd),
// finalisation, the on-request 5-D pair mask, the bf16 hi/lo operand pack and the backward scales.
// Reference: utils/utils.py:779-893 (descriptor_loss), :745-768 (normPts/denormPts), :315-343.
#include "desc_common.cuh"
#include <cuda_bf16.h>

// ----------------------------------------------------------------------------------------------
// geometry: warped cell centres  w = denorm(swap(warp(swap(norm(c)))))   [utils/utils.py:829-851]
// ----------------------------------------------------------------------------------------------
// mask_valid [B, Nc] (cell resolution) or, when it is NULL, mask2d [B, 1, 8 Hc, 8 Wc]: the cell mask is then the product of
// the 64 sub-pixels of every cell, in the order of getMasks / cell_mask_kernel (Train_model_frontend_all.py:373-386).
struct GeomArgs {
  const float* Hm; const float* mask_valid; const float* mask2d; int B, Hc, Wc, cell, Nc_pad;
  float2* wpts; float* mv_pad; double* mv_part; uint32_t* mvbits;
};
#define GEOM_THREADS 256
// (bx, by) = block coordinates in a (Nc_pad / GEOM_THREADS, B) grid; shd: >= 32 doubles of shared memory
__device__ __forceinline__ void desc_geometry_block(const GeomArgs& A, int bx, int by, int gridx, double* shd) {
  const float* __restrict__ Hm = A.Hm; const float* __restrict__ mask_valid = A.mask_valid;
  const float* __restrict__ mask2d = A.mask2d;
  const int Hc = A.Hc, Wc = A.Wc, cell = A.cell, Nc_pad = A.Nc_pad;
  float2* __restrict__ wpts = A.wpts; float* __restrict__ mv_pad = A.mv_pad; double* __restrict__ mv_part = A.mv_part;
  uint32_t* __restrict__ mvbits = A.mvbits;
  int b = by;
  int c = bx * blockDim.x + threadIdx.x;  // Nc_pad is a multiple of the block size
  int Nc = Hc * Wc;
  float2 w = make_float2(SSP_FAR, SSP_FAR);
  float mv = 0.f;
  if (c < Nc) {
    float cx, cy;
    cell_center(c, Wc, cell, cx, cy);
    float Hpx = (float)(Hc * cell), Wpx = (float)(Wc * cell);
    // normPts divides by (H, W), not (H-1, W-1)   [utils/utils.py:745-755, :838]
    float ny = cy / Hpx * 2.f - 1.f;
    float nx = cx / Wpx * 2.f - 1.f;
    float ox, oy;
    homography_apply(Hm + b * 9, nx, ny, ox, oy);
    // denormPts: (p + 1) * shape / 2   [utils/utils.py:758-768]
    w.x = (ox + 1.f) * Wpx / 2.f;
    w.y = (oy + 1.f) * Hpx / 2.f;
    mv = mask_valid ? mask_valid[(size_t)b * Nc + c] : 1.f;
    if (!mask_valid && mask2d) {
      const int W = Wc * 8;
      const float* img = mask2d + (size_t)b * Nc * 64 + (size_t)((c / Wc) * 8) * W + (c % Wc) * 8;
      float p = 1.f;
      bool first = true;
#pragma unroll
      for (int dy = 0; dy < 8; ++dy) {
        const float4* r = reinterpret_cast<const float4*>(img + (size_t)dy * W);
        const float4 a = __ldg(r), q = __ldg(r + 1);
        const float v[8] = {a.x, a.y, a.z, a.w, q.x, q.y, q.z, q.w};
#pragma unroll
        for (int dx = 0; dx < 8; ++dx) {
          p = first ? v[dx] : p * v[dx];
          first = false;
        }
      }
      mv = p;
    }
  }
  wpts[(size_t)b * Nc_pad + c] = w;
  mv_pad[(size_t)b * Nc_pad + c] = mv;
  double mvs = (double)mv;
  if (mvbits) {
    // "fold" mode of the tensor-core engine: the mask is folded into the indicator words, which is only exact for a
    // BINARY mask.  Anything else poisons the normaliser (NaN loss and gradients): loud, and without a host sync.
    if (mv != 0.f && mv != 1.f) mvs = __longlong_as_double(0x7ff8000000000000ll);
    const uint32_t word = __reduce_or_sync(0xffffffffu, (mv != 0.f ? 1u : 0u) << DESC_BITPOS(threadIdx.x & 31));
    if ((threadIdx.x & 31) == 0) mvbits[((size_t)b * Nc_pad + c) >> 5] = word;
  }
  // per-block partial of sum(mask_valid) for the global normaliser (summed in fixed order by finalize)
  double part = block_sum_d(mvs, shd);
  if (threadIdx.x == 0) mv_part[(size_t)b * gridx + bx] = part;
}

__global__ void __launch_bounds__(GEOM_THREADS) desc_geometry_kernel(const __grid_constant__ GeomArgs A) {
  __shared__ double shd[32];
  desc_geometry_block(A, blockIdx.x, blockIdx.y, gridDim.x, shd);
}

extern "C" int ssp_desc_geometry_nblocks(int B, int Nc) { return B * (desc_nc_pad(Nc) / GEOM_THREADS); }

// candidate window of cell indices whose centre can be within `dist` of (wx, wy): a centre k*cell + half qualifies only if
// |k*cell + half - w| <= dist, i.e. k in [(w - dist - half)/cell, (w + dist - half)/cell]; the window is that interval
// widened by 0.01 cell (0.08 px at cell = 8: three orders of magnitude above the fp32 rounding of pixel coordinates), the
// exact predicate decides.  <= 2 x 2 candidates for dist <= cell/2, <= 3 x 3 for dist <= cell (it used to be 5 x 5, and
// the scan was two thirds of the instructions of the pos kernels).
__device__ __forceinline__ void pos_window(float wx, float wy, float dist, int Hc, int Wc, int cell, int& k0,
                                           int& k1, int& l0, int& l1) {
  float half = (float)(cell / 2), fc = (float)cell;
  float a = ceilf((wy - dist - half) / fc - 0.01f), b = floorf((wy + dist - half) / fc + 0.01f);
  float c = ceilf((wx - dist - half) / fc - 0.01f), d = floorf((wx + dist - half) / fc + 0.01f);
  // clamp in float first: far-away / non-finite points give an empty window
  k0 = (int)fmaxf(a, 0.f);
  k1 = (int)fminf(b, (float)(Hc - 1));
  l0 = (int)fmaxf(c, 0.f);
  l1 = (int)fminf(d, (float)(Wc - 1));
  if (!(a <= (float)Hc && b >= -1.f && c <= (float)Wc && d >= -1.f)) { k0 = 1; k1 = 0; }
}

// ----------------------------------------------------------------------------------------------
// positive pairs, forward.  The dense GEMM kernel treats EVERY pair as a negative (no geometry in its
// epilogue); this kernel owns the sparse positive set (<= DESC_MAXP per row for descriptor_dist <= cell):
//   * exact fp32 dot product of every positive pair (block = 32 rows x 8 channel groups, coalesced in NCHW)
//   * partial sums  lamda*max(mpos-dot,0)  and the correction  max(dot-mneg,0)  that the dense sum wrongly
//     contains for these pairs (the hinge is continuous, so the mismatch between this exact dot and the
//     tensor-core dot is bounded by their difference, ~1e-6)
//   * pair lists for the backward: per row (partner column, dot) and, through an atomic slot counter, per
//     column (partner row, dot)
// partials: 4 doubles per block = { pos_unweighted, pos_weighted, negcorr_unweighted, negcorr_weighted }
// ----------------------------------------------------------------------------------------------
// Latency chain per block (the kernel is latency-bound: 1280 blocks of short dependent steps): geometry scan ->
// one round of loads covering TWO partners per row (rows have 0.8 partners on average, rarely more than 2) -> one
// shared-memory combine -> list stores / slot atomics fired by warp 0 without anybody waiting on them -> warp-level
// reduction of the four partial sums.
#define POS_ROWS 32
#define POS_DG 8
#define POS_CH 16  // channels per thread and chunk (3 x 16 independent loads in flight)
__global__ void __launch_bounds__(POS_ROWS * POS_DG, 2)
desc_pos_fwd_kernel(const float* __restrict__ D, const float* __restrict__ Dw, const float2* __restrict__ wpts,
                    const float* __restrict__ mv_pad, DescGeom g, double* __restrict__ partials,
                    int* __restrict__ rowcol, float* __restrict__ rowdot, int* __restrict__ colcnt,
                    int* __restrict__ colrow, float* __restrict__ coldot) {
  __shared__ int scol[POS_ROWS][DESC_MAXP];
  __shared__ int scnt[POS_ROWS];
  __shared__ float spart[2][POS_DG][POS_ROWS];
  __shared__ int smax;
  const int b = blockIdx.y, lane = threadIdx.x & 31, dg = threadIdx.x >> 5;
  const int r = blockIdx.x * POS_ROWS + lane;
  if (threadIdx.x == 0) smax = 0;
  __syncthreads();
  if (dg == 0) {
    int cnt = 0;
    if (r < g.Nc) {
      float2 w = wpts[(size_t)b * g.Nc_pad + r];
      int k0, k1, l0, l1;
      pos_window(w.x, w.y, g.dist, g.Hc, g.Wc, g.cell, k0, k1, l0, l1);
      int dropped = 0;
      for (int k = k0; k <= k1; ++k)
        for (int l = l0; l <= l1; ++l) {
          int c = k * g.Wc + l;
          float cx, cy;
          cell_center(c, g.Wc, g.cell, cx, cy);
          if (pair_positive(w.x, w.y, cx, cy, g.dist)) {
            if (cnt < DESC_MAXP) scol[lane][cnt++] = c;
            else ++dropped;
          }
        }
      if (dropped) atomicAdd(colcnt + (size_t)g.B * g.Nc_pad, dropped);  // overflow counter: finalize turns it into NaN
    }
    scnt[lane] = cnt;
    if (r < g.Nc_pad) {
      int4* rc = reinterpret_cast<int4*>(rowcol + ((size_t)b * g.Nc_pad + r) * DESC_MAXP);
#pragma unroll
      for (int n = 0; n < DESC_MAXP; n += 4)
        rc[n / 4] = make_int4(n < cnt ? scol[lane][n] : -1, n + 1 < cnt ? scol[lane][n + 1] : -1,
                              n + 2 < cnt ? scol[lane][n + 2] : -1, n + 3 < cnt ? scol[lane][n + 3] : -1);
    }
    if (cnt) atomicMax(&smax, cnt);
  }
  __syncthreads();
  const int nmax = smax;
  const int cnt = scnt[lane];
  const int dper = (g.Dch + POS_DG - 1) / POS_DG;
  const int d0 = dg * dper, d1 = min(g.Dch, d0 + dper);
  const float* __restrict__ Db = D + (size_t)b * g.Dch * g.Nc + r;
  const float* __restrict__ Dwb = Dw + (size_t)b * g.Dch * g.Nc;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int n0 = 0; n0 < nmax; n0 += 2) {
    const bool has0 = n0 < cnt, has1 = n0 + 1 < cnt;
    const int c0 = has0 ? scol[lane][n0] : 0, c1 = has1 ? scol[lane][n0 + 1] : 0;
    float part0 = 0.f, part1 = 0.f;
    if (has0) {
      for (int db = d0; db < d1; db += POS_CH) {
        float a[POS_CH], w0[POS_CH], w1[POS_CH];
#pragma unroll
        for (int i = 0; i < POS_CH; ++i) {
          bool ok = db + i < d1;
          a[i] = ok ? __ldg(Db + (size_t)(db + i) * g.Nc) : 0.f;
          w0[i] = ok ? __ldg(Dwb + (size_t)(db + i) * g.Nc + c0) : 0.f;
          w1[i] = (ok && has1) ? __ldg(Dwb + (size_t)(db + i) * g.Nc + c1) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < POS_CH; ++i) {
          part0 = fmaf(a[i], w0[i], part0);
          part1 = fmaf(a[i], w1[i], part1);
        }
      }
    }
    if (n0) __syncthreads();  // warp 0 has consumed the previous round
    spart[0][dg][lane] = part0;
    spart[1][dg][lane] = part1;
    __syncthreads();
    if (dg == 0) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (!(j ? has1 : has0)) continue;
        const int c = j ? c1 : c0;
        float dot = 0.f;
#pragma unroll
        for (int q = 0; q < POS_DG; ++q) dot += spart[j][q][lane];
        float mv = mv_pad[(size_t)b * g.Nc_pad + c];
        float pos = g.lamda * fmaxf(g.mpos - dot, 0.f);
        float negc = fmaxf(dot - g.mneg, 0.f);
        acc[0] += (double)pos;
        acc[1] += (double)(pos * mv);
        acc[2] += (double)negc;
        acc[3] += (double)(negc * mv);
        rowdot[((size_t)b * g.Nc_pad + r) * DESC_MAXP + n0 + j] = dot;
        int slot = atomicAdd(colcnt + (size_t)b * g.Nc_pad + c, 1);
        if (slot < DESC_MAXP) {
          colrow[((size_t)b * g.Nc_pad + c) * DESC_MAXP + slot] = r;
          coldot[((size_t)b * g.Nc_pad + c) * DESC_MAXP + slot] = dot;
        } else {
          atomicAdd(colcnt + (size_t)g.B * g.Nc_pad, 1);  // overflow counter
        }
      }
    }
  }
  if (dg == 0) {  // only warp 0 holds sums
    size_t blk = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double v = warp_sum_d(acc[i]);
      if (lane == 0) partials[4 * blk + i] = v;
    }
  }
}

// the grid covers all Nc_pad rows so that every list row is initialised (padded rows get empty lists)
extern "C" int ssp_desc_pos_nblocks(int B, int Nc) { return B * (desc_nc_pad(Nc) / POS_ROWS); }
extern "C" int ssp_desc_maxp(void) { return DESC_MAXP; }

static int fill_geom(DescGeom& g, int B, int Hc, int Wc, int Dch, int cell, float dist, float lamda, float mpos,
                     float mneg) {
  g.B = B; g.Hc = Hc; g.Wc = Wc; g.Nc = Hc * Wc; g.Nc_pad = desc_nc_pad(Hc * Wc); g.Dch = Dch;
  g.cell = cell; g.dist = dist; g.lamda = lamda; g.mpos = mpos; g.mneg = mneg;
  return (B > 0 && Hc > 0 && Wc > 0 && Dch > 0 && cell > 0) ? 0 : -1;
}

// Lists: rowcol/rowdot/colrow/coldot [B, Nc_pad, DESC_MAXP], colcnt [B*Nc_pad + 1] (zeroed here; the last
// element counts pairs that did not fit a column list).
extern "C" int ssp_desc_pos_fwd(const float* D, const float* Dw, const float* wpts, const float* mv_pad, int B,
                                int Hc, int Wc, int Dch, int cell, float dist, float lamda, float mpos, float mneg,
                                double* partials, int* rowcol, float* rowdot, int* colcnt, int* colrow,
                                float* coldot, void* stream) {
  SSP_REQUIRE(D && Dw && wpts && mv_pad && partials && rowcol && rowdot && colcnt && colrow && coldot,
              "ssp_desc_pos_fwd: null pointer");
  DescGeom g;
  SSP_REQUIRE(fill_geom(g, B, Hc, Wc, Dch, cell, dist, lamda, mpos, mneg) == 0 && B <= 65535, "ssp_desc_pos_fwd: bad sizes");
  SSP_REQUIRE(dist >= 0.f && dist <= (float)cell,
              "ssp_desc_pos_fwd: descriptor_dist %.3f > cell_size %d is not supported (sparse positive lists hold %d pairs per cell)",
              dist, cell, DESC_MAXP);
  cudaStream_t st = (cudaStream_t)stream;
  SSP_CUDA_CALL(cudaMemsetAsync(colcnt, 0, ((size_t)B * g.Nc_pad + 1) * sizeof(int), st));
  dim3 grid(g.Nc_pad / POS_ROWS, B);
  desc_pos_fwd_kernel<<<grid, POS_ROWS * POS_DG, 0, st>>>(D, Dw, reinterpret_cast<const float2*>(wpts), mv_pad, g,
                                                           partials, rowcol, rowdot, colcnt, colrow, coldot);
  SSP_CUDA_CHECK_LAUNCH("desc_pos_fwd_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// positive pairs, forward, from the PACKED planes (bf16x3 engine).  NCHW keeps the 256 channels of a cell 4.8 KB
// apart, so the kernel above pays one 32 B sector (and one L1 wavefront) per channel per gathered partner; the
// [cell][256] hi/lo planes that the tensor-core kernels consume hold a cell's descriptor as 2 x 512 contiguous bytes.
// One warp per row: lanes test the candidate window in parallel (ballot compaction keeps the k-major, l-minor order
// of the sequential scan), then every partner costs four fully coalesced 512 B loads and a warp reduction.
// hi + lo carries 16 mantissa bits (relative error 2^-17 per element): the dot is as accurate as the bf16x3 GEMM's own
// value for the pair, which is what the negative-hinge correction must cancel.
// partials: 4 doubles per block, as above.  Same lists.
// ----------------------------------------------------------------------------------------------
#define POSP_ROWS 64      // rows per block
#define POSP_THREADS 256  // phase 2: 8 lanes per row, 32 rows per pass
__device__ __forceinline__ void bf16x8_sum(const uint4& h, const uint4& l, float (&v)[8]) {
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
    v[2 * i + 1] = __uint_as_float(hw[i] & 0xffff0000u) + __uint_as_float(lw[i] & 0xffff0000u);
  }
}

// Block = 64 rows.  Phase 1: one thread per row scans its candidate window sequentially (k-major, l-minor: the order of
// the lists) -- a few cells for descriptor_dist <= cell.  Phase 2: EIGHT lanes per row, each covering 32 channels = 4 + 4
// 16-byte loads per side, all 16 issued before the first use: the kernel is a chain of dependent latencies (point ->
// window -> partner -> planes -> atomics), so what matters is how many bytes every warp has in flight (8 KB here; the
// previous one-warp-per-row version had 1 KB and ran at 27 us for 150 MB of L2-resident planes).
__global__ void __launch_bounds__(POSP_THREADS)
desc_pos_fwd_planes_kernel(const uint4* __restrict__ Ahi, const uint4* __restrict__ Alo, const uint4* __restrict__ Bhi,
                           const uint4* __restrict__ Blo, const float2* __restrict__ wpts,
                           const float* __restrict__ mv_pad, DescGeom g, double* __restrict__ partials,
                           int* __restrict__ rowcol, float* __restrict__ rowdot, int* __restrict__ colcnt,
                           int* __restrict__ colrow, float* __restrict__ coldot) {
  __shared__ int scol[POSP_ROWS][DESC_MAXP + 1];
  __shared__ int scnt[POSP_ROWS];
  __shared__ double sred[32];
  const int tid = threadIdx.x;
  const int b = blockIdx.y, r0 = blockIdx.x * POSP_ROWS;  // grid.x covers Nc_pad rows
  if (tid < POSP_ROWS) {
    const int r = r0 + tid;
    int cnt = 0;
    if (r < g.Nc) {
      const float2 w = wpts[(size_t)b * g.Nc_pad + r];
      int k0, k1, l0, l1;
      pos_window(w.x, w.y, g.dist, g.Hc, g.Wc, g.cell, k0, k1, l0, l1);
      int dropped = 0;
      for (int k = k0; k <= k1; ++k)
        for (int l = l0; l <= l1; ++l) {
          const int c = k * g.Wc + l;
          float cx, cy;
          cell_center(c, g.Wc, g.cell, cx, cy);
          if (pair_positive(w.x, w.y, cx, cy, g.dist)) {
            if (cnt < DESC_MAXP) scol[tid][cnt++] = c;
            else ++dropped;
          }
        }
      if (dropped) atomicAdd(colcnt + (size_t)g.B * g.Nc_pad, dropped);  // overflow counter: finalize turns it into NaN
    }
    scnt[tid] = cnt;
    int4* rc = reinterpret_cast<int4*>(rowcol + ((size_t)b * g.Nc_pad + r) * DESC_MAXP);
#pragma unroll
    for (int n = 0; n < DESC_MAXP; n += 4)
      rc[n / 4] = make_int4(n < cnt ? scol[tid][n] : -1, n + 1 < cnt ? scol[tid][n + 1] : -1,
                            n + 2 < cnt ? scol[tid][n + 2] : -1, n + 3 < cnt ? scol[tid][n + 3] : -1);
  }
  __syncthreads();
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int sub = tid & 7;  // lane within the row's group of eight: channels [32 sub, 32 sub + 32)
#pragma unroll 1
  for (int pass = 0; pass < POSP_ROWS / 32; ++pass) {
    const int lr = pass * 32 + (tid >> 3), r = r0 + lr;
    const int cnt = scnt[lr];
    if (cnt == 0) continue;  // the eight lanes of a group agree; shuffles below stay inside the group
    const unsigned gmask = 0xFFu << ((tid & 31) & ~7);
    const uint4* pa_h = Ahi + ((size_t)b * g.Nc_pad + r) * 32 + sub * 4;
    const uint4* pa_l = Alo + ((size_t)b * g.Nc_pad + r) * 32 + sub * 4;
    uint4 ah[4], al[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) { ah[t] = __ldg(pa_h + t); al[t] = __ldg(pa_l + t); }
    for (int n = 0; n < cnt; ++n) {
      const int c = scol[lr][n];
      const uint4* pb_h = Bhi + ((size_t)b * g.Nc_pad + c) * 32 + sub * 4;
      const uint4* pb_l = Blo + ((size_t)b * g.Nc_pad + c) * 32 + sub * 4;
      uint4 bh[4], bl[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) { bh[t] = __ldg(pb_h + t); bl[t] = __ldg(pb_l + t); }
      float part = 0.f;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float a[8], w8[8];
        bf16x8_sum(ah[t], al[t], a);
        bf16x8_sum(bh[t], bl[t], w8);
#pragma unroll
        for (int i = 0; i < 8; ++i) part = fmaf(a[i], w8[i], part);
      }
      part += __shfl_xor_sync(gmask, part, 4);
      part += __shfl_xor_sync(gmask, part, 2);
      part += __shfl_xor_sync(gmask, part, 1);
      if (sub == 0) {
        const float dot = part;
        const float mv = mv_pad[(size_t)b * g.Nc_pad + c];
        const float pos = g.lamda * fmaxf(g.mpos - dot, 0.f);
        const float negc = fmaxf(dot - g.mneg, 0.f);
        acc[0] += (double)pos;
        acc[1] += (double)(pos * mv);
        acc[2] += (double)negc;
        acc[3] += (double)(negc * mv);
        rowdot[((size_t)b * g.Nc_pad + r) * DESC_MAXP + n] = dot;
        const int slot = atomicAdd(colcnt + (size_t)b * g.Nc_pad + c, 1);
        if (slot < DESC_MAXP) {
          colrow[((size_t)b * g.Nc_pad + c) * DESC_MAXP + slot] = r;
          coldot[((size_t)b * g.Nc_pad + c) * DESC_MAXP + slot] = dot;
        } else {
          atomicAdd(colcnt + (size_t)g.B * g.Nc_pad, 1);  // overflow counter
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double v = block_sum_d(acc[i], sred);  // fixed tree: deterministic
    if (tid == 0) partials[4 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x) + i] = v;
  }
}

extern "C" int ssp_desc_pos_planes_nblocks(int B, int Nc) { return B * (desc_nc_pad(Nc) / POSP_ROWS); }

// Same contract as ssp_desc_pos_fwd, reading the packed hi/lo planes [B, Nc_pad, 256] of D (A*) and Dw (B*).
extern "C" int ssp_desc_pos_fwd_planes(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo,
                                       const float* wpts, const float* mv_pad, int B, int Hc, int Wc, int cell, float dist,
                                       float lamda, float mpos, float mneg, double* partials, int* rowcol, float* rowdot,
                                       int* colcnt, int* colrow, float* coldot, void* stream) {
  SSP_REQUIRE(Ahi && Alo && Bhi && Blo && wpts && mv_pad && partials && rowcol && rowdot && colcnt && colrow && coldot,
              "ssp_desc_pos_fwd_planes: null pointer");
  SSP_REQUIRE(((((uintptr_t)Ahi | (uintptr_t)Alo | (uintptr_t)Bhi | (uintptr_t)Blo) & 15) == 0),
              "ssp_desc_pos_fwd_planes: planes must be 16-byte aligned");
  DescGeom g;
  SSP_REQUIRE(fill_geom(g, B, Hc, Wc, 256, cell, dist, lamda, mpos, mneg) == 0 && B <= 65535, "ssp_desc_pos_fwd_planes: bad sizes");
  SSP_REQUIRE(dist >= 0.f && dist <= (float)cell,
              "ssp_desc_pos_fwd_planes: descriptor_dist %.3f > cell_size %d is not supported (sparse positive lists hold %d pairs per cell)",
              dist, cell, DESC_MAXP);
  cudaStream_t st = (cudaStream_t)stream;
  SSP_CUDA_CALL(cudaMemsetAsync(colcnt, 0, ((size_t)B * g.Nc_pad + 1) * sizeof(int), st));
  dim3 grid(g.Nc_pad / POSP_ROWS, B);
  desc_pos_fwd_planes_kernel<<<grid, POSP_THREADS, 0, st>>>(
      (const uint4*)Ahi, (const uint4*)Alo, (const uint4*)Bhi, (const uint4*)Blo, reinterpret_cast<const float2*>(wpts), mv_pad, g,
      partials, rowcol, rowdot, colcnt, colrow, coldot);
  SSP_CUDA_CHECK_LAUNCH("desc_pos_fwd_planes_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// finalize: fixed-order sums of the partials, global-batch normaliser  [utils/utils.py:883-890]
//   out8 = { loss_desc, pos_sum, neg_sum, normalization, num_loss, num_pos, num_neg, sum(mask_valid) }
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
desc_finalize_kernel(const double* __restrict__ pos_part, int npos, const double* __restrict__ neg_part, int nneg,
                     const double* __restrict__ mv_part, int nmv, int B, int Hc, int Wc, const int* __restrict__ overflow,
                     float* __restrict__ out4, const float* __restrict__ det0, const float* __restrict__ det1,
                     float lambda_loss, float* __restrict__ total) {
  __shared__ double sh[7][32];
  double pu = 0, pw = 0, nu = 0, nw = 0, sm = 0;
  double cu = 0, cw = 0;  // negative-hinge contribution of the positive pairs, contained in the dense sums
  // One block, so the kernel is a chain of L2 round trips unless the loads of all three arrays are in flight together:
  // the first batch of each array is issued before anything is summed (at the headline sizes there is no second batch).
  const double2* p2 = reinterpret_cast<const double2*>(pos_part);  // {pos_u, pos_w}, {negcorr_u, negcorr_w}
  const double2* n2 = reinterpret_cast<const double2*>(neg_part);
  const int T = blockDim.x, t = threadIdx.x;
  const double2 z2 = make_double2(0.0, 0.0);
  for (int base = 0; base < npos || base < nneg || base < nmv; base += 2 * T) {
    double2 a[2], c[2], n[2];
    double m[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = base + u * T + t;
      a[u] = i < npos ? p2[2 * (size_t)i] : z2;
      c[u] = i < npos ? p2[2 * (size_t)i + 1] : z2;
      n[u] = i < nneg ? n2[i] : z2;
      m[u] = i < nmv ? mv_part[i] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      pu += a[u].x; pw += a[u].y; cu += c[u].x; cw += c[u].y; nu += n[u].x; nw += n[u].y; sm += m[u];
    }
  }
  // seven block sums behind ONE pair of barriers (fixed tree: deterministic)
  {
    double v[7] = {pu, pw, nu, nw, sm, cu, cw};
    const int lane = t & 31, w = t >> 5, nwarps = (T + 31) >> 5;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      v[k] = warp_sum_d(v[k]);
      if (lane == 0) sh[k][w] = v[k];
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
      for (int k = 0; k < 7; ++k) v[k] = warp_sum_d(lane < nwarps ? sh[k][lane] : 0.0);
    }
    pu = v[0]; pw = v[1]; nu = v[2]; nw = v[3]; sm = v[4]; cu = v[5]; cw = v[6];
  }
  if (threadIdx.x == 0) {
    nu -= cu;
    nw -= cw;
    // positive pairs that did not fit the sparse lists (strong minification, descriptor_dist close to the cell size): the
    // loss and its gradient would silently miss them -- poison the result instead (NaN, no host sync needed to notice)
    if (overflow && *overflow != 0) pu = pw = __longlong_as_double(0x7ff8000000000000ll);
    float norm = (float)B * ((float)sm + 1.f) * (float)Hc * (float)Wc;
    out4[0] = (float)((pw + nw) / (double)norm);
    out4[1] = (float)(pu / (double)norm);
    out4[2] = (float)(nu / (double)norm);
    out4[3] = norm;
    // raw sums for the multi-GPU exchange (global-batch normaliser, SURVEY 8e)
    out4[4] = (float)(pw + nw);
    out4[5] = (float)pu;
    out4[6] = (float)nu;
    out4[7] = (float)sm;
    // fused loss step: total = loss_det + loss_det_warp + lambda_loss * loss_desc (Train_model_heatmap_all.py:361-365),
    // same fp32 operation order as the torch expression it replaces
    if (total) *total = (det0[0] + det1[0]) + lambda_loss * out4[0];
  }
}

// overflow (optional): the list-overflow counter colcnt[B * Nc_pad] of the pos kernels; non-zero poisons loss and pos with NaN.
// total (optional, with det0 / det1 = the out3 triples of the two detector losses): the weighted sum of the fused loss step.
extern "C" int ssp_desc_finalize(const double* pos_part, int npos, const double* neg_part, int nneg,
                                 const double* mv_part, int nmv, int B, int Hc, int Wc, const int* overflow, float* out4,
                                 const float* det0, const float* det1, float lambda_loss, float* total, void* stream) {
  SSP_REQUIRE(pos_part && neg_part && mv_part && out4, "ssp_desc_finalize: null pointer");
  SSP_REQUIRE(npos >= 0 && nneg >= 0 && nmv >= 0 && B > 0 && Hc > 0 && Wc > 0, "ssp_desc_finalize: bad sizes");
  SSP_REQUIRE((((uintptr_t)pos_part | (uintptr_t)neg_part) & 15) == 0, "ssp_desc_finalize: partial-sum arrays must be 16-byte aligned");
  SSP_REQUIRE(!total || (det0 && det1), "ssp_desc_finalize: the step total needs both detector triples");
  desc_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(pos_part, npos, neg_part, nneg, mv_part, nmv, B, Hc, Wc, overflow, out4,
                                                             det0, det1, lambda_loss, total);
  SSP_CUDA_CHECK_LAUNCH("desc_finalize_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// the 5-D correspondence mask [B,Hc,Wc,Hc,Wc] (float 0/1) -- returned by the reference but never read
// by its caller; materialised only on request.
// ----------------------------------------------------------------------------------------------
__global__ void desc_pair_mask_kernel(const float2* __restrict__ wpts, DescGeom g, float* __restrict__ mask) {
  int b = blockIdx.z, r = blockIdx.y;
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= g.Nc) return;
  float2 w = wpts[(size_t)b * g.Nc_pad + r];
  float cx, cy;
  cell_center(c, g.Wc, g.cell, cx, cy);
  mask[((size_t)b * g.Nc + r) * g.Nc + c] = pair_positive(w.x, w.y, cx, cy, g.dist) ? 1.f : 0.f;
}

extern "C" int ssp_desc_pair_mask(const float* wpts, int B, int Hc, int Wc, int cell, float dist, float* mask,
                                  void* stream) {
  SSP_REQUIRE(wpts && mask, "ssp_desc_pair_mask: null pointer");
  DescGeom g;
  SSP_REQUIRE(fill_geom(g, B, Hc, Wc, 1, cell, dist, 0.f, 0.f, 0.f) == 0 && B <= 65535 && g.Nc <= 65535,
              "ssp_desc_pair_mask: bad sizes");
  dim3 grid(ssp_ceil_div(g.Nc, 256), g.Nc, B);
  desc_pair_mask_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(wpts), g, mask);
  SSP_CUDA_CHECK_LAUNCH("desc_pair_mask_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// backward scales: alpha[b,c] = (g_loss * mv[b,c] + g_neg) / norm   (coefficient of the negative hinge)
// ----------------------------------------------------------------------------------------------
__global__ void desc_alpha_kernel(const float* __restrict__ mv_pad, const float* __restrict__ g3,
                                  const float* __restrict__ out4, size_t n, float* __restrict__ alpha) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) alpha[i] = (g3[0] * mv_pad[i] + g3[2]) / out4[3];
}

extern "C" int ssp_desc_alpha(const float* mv_pad, const float* g3, const float* out4, int B, int Nc_pad, float* alpha,
                              void* stream) {
  SSP_REQUIRE(mv_pad && g3 && out4 && alpha, "ssp_desc_alpha: null pointer");
  size_t n = (size_t)B * Nc_pad;
  desc_alpha_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mv_pad, g3, out4, n, alpha);
  SSP_CUDA_CHECK_LAUNCH("desc_alpha_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// positive pairs, backward: per-list-entry coefficients consumed by the indicator-GEMM epilogues.
//   coef = -lamda * ind(mpos - dot) * (g_loss * mv[c] + g_pos) / norm,  ind = 1 (x>0), 0.5 (x==0), 0 (x<0)
//          - (bit(r,c) ? alpha[c] : 0)        <- removes the negative-hinge term the indicator GEMM adds for
//                                                this pair (its bit is set whenever the dense dot exceeded mneg)
//   rows: rowcoef[b,r,n] for partner column rowcol[b,r,n]          (dD [b,:,r] += coef * Dw[b,:,c])
//   cols: entries sorted by row index (deterministic sum order), colcoef (dDw[b,:,c] += coef * D [b,:,r])
// ----------------------------------------------------------------------------------------------
#include "desc_pos_coef.cuh"

__global__ void __launch_bounds__(128) desc_pos_coef_kernel(const __grid_constant__ PosCoefArgs A) {
  desc_pos_coef_block(A, blockIdx.x, blockIdx.y, blockIdx.z, gridDim.x);
}

// alpha_out (optional, [B, Nc_pad]): the vector ssp_desc_alpha would write for the same (scaled) gradients -- the fused step
// gets it from this launch and skips that kernel; srow_out (optional, [B, Nc_pad]): the same coefficient at mask_valid = 1,
// the row scale of the folded backward (mask already inside the bits).
// bitsC_out (optional, with Nc = the unpadded cell count): the column-orientation indicator words, transposed from bitsR by
// extra blocks of the same launch (the tensor-core forward then needs no transpose kernel).
extern "C" int ssp_desc_pos_coef(const int* rowcol, const float* rowdot, const int* colcnt, const int* colrow,
                                 const float* coldot, const uint32_t* bitsR, const float* mv_pad, const float* g3, float gscale,
                                 int gmode, const float* out8, int B, int Nc_pad, float lamda, float mpos, float* rowcoef,
                                 int* colrow_sorted, float* colcoef, float* alpha_out, float* srow_out, uint32_t* bitsC_out,
                                 int Nc, void* stream) {
  SSP_REQUIRE(rowcol && rowdot && colcnt && colrow && coldot && bitsR && mv_pad && g3 && out8 && rowcoef && colrow_sorted && colcoef,
              "ssp_desc_pos_coef: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Nc_pad > 0 && Nc_pad % DESC_PAD == 0 && (gmode == 0 || gmode == 1), "ssp_desc_pos_coef: bad sizes");
  SSP_REQUIRE(!bitsC_out || (Nc > 0 && Nc <= Nc_pad), "ssp_desc_pos_coef: bitsC_out needs the cell count Nc");
  dim3 grid(ssp_ceil_div(Nc_pad, 128), B, bitsC_out ? 6 : 2);
  PosCoefArgs A = {rowcol, rowdot, colcnt, colrow, coldot, bitsR, mv_pad, g3, gscale, gmode, out8, Nc_pad, lamda, mpos,
                   rowcoef, colrow_sorted, colcoef, alpha_out, srow_out, bitsC_out, (Nc + 31) / 32};
  desc_pos_coef_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(A);
  SSP_CUDA_CHECK_LAUNCH("desc_pos_coef_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// positive pairs, backward apply: out[b, d, r] += sum_n coef[b, r, n] * src[b, d, list[b, r, n]]
// for both gradients in one launch (blockIdx.z = 0: dD with Dw as src, 1: dDw with D as src).  Streaming
// kernel, every access is a 128 B line per warp (list partners of neighbouring cells are neighbours).  Runs after the indicator GEMMs stored dD / dDw.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
desc_pos_apply_kernel(const int* __restrict__ rowcol, const float* __restrict__ rowcoef, const int* __restrict__ colrow,
                      const float* __restrict__ colcoef, const float* __restrict__ D, const float* __restrict__ Dw,
                      int Dch, int Nc, int Nc_pad, float* __restrict__ dD, float* __restrict__ dDw) {
  // block = 128 consecutive cells x 2 sub-groups of 16 channels: 512 contiguous bytes per channel row per block
  const int b = blockIdx.y;
  const int r = blockIdx.x * 128 + (threadIdx.x & 127), sub = threadIdx.x >> 7;
  const int nd32 = (Dch + 31) / 32;
  const bool second = (int)blockIdx.z >= nd32;
  const int d0 = ((int)blockIdx.z % nd32) * 32 + sub * 16;
  if (r >= Nc || d0 >= Dch) return;
  const int* list = (second ? colrow : rowcol) + ((size_t)b * Nc_pad + r) * DESC_MAXP;
  const float* coef = (second ? colcoef : rowcoef) + ((size_t)b * Nc_pad + r) * DESC_MAXP;
  const float* src = (second ? D : Dw) + ((size_t)b * Dch + d0) * Nc;
  float* out = (second ? dDw : dD) + ((size_t)b * Dch + d0) * Nc + r;
  const int nd = min(16, Dch - d0);
  for (int n = 0; n < DESC_MAXP; ++n) {
    int pc = list[n];
    if (pc < 0) break;  // lists are filled front to back
    float cf = coef[n];
    if (cf == 0.f) continue;
    float o[16], v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {  // all loads issued before the first store
      o[i] = i < nd ? out[(size_t)i * Nc] : 0.f;
      v[i] = i < nd ? __ldg(src + (size_t)i * Nc + pc) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < nd) out[(size_t)i * Nc] = fmaf(cf, v[i], o[i]);
  }
}

extern "C" int ssp_desc_pos_apply(const int* rowcol, const float* rowcoef, const int* colrow, const float* colcoef,
                                  const float* D, const float* Dw, int B, int Dch, int Nc, float* dD, float* dDw,
                                  void* stream) {
  SSP_REQUIRE(rowcol && rowcoef && colrow && colcoef && D && Dw && dD && dDw, "ssp_desc_pos_apply: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Dch > 0 && Nc > 0, "ssp_desc_pos_apply: bad sizes");
  dim3 grid(ssp_ceil_div(Nc, 128), B, 2 * ssp_ceil_div(Dch, 32));
  desc_pos_apply_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rowcol, rowcoef, colrow, colcoef, D, Dw, Dch, Nc,
                                                                desc_nc_pad(Nc), dD, dDw);
  SSP_CUDA_CHECK_LAUNCH("desc_pos_apply_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// operand pack for the tcgen05 engine: [B, Dch, Nc] fp32 (NCHW) -> K-major bf16 planes
//   hi[b, c, d] = bf16(s * x),  lo[b, c, d] = bf16(s * x - hi)   (lo optional), rows c >= Nc zeroed
//   s = scale[b, c] if given (backward: alpha), else 1.
// 32 cells x Dch tile transposed through shared memory; reads are 128 B per warp per channel, writes
// are contiguous bf16 rows.
// ----------------------------------------------------------------------------------------------
#define PK_CELLS 64   // cells per block: 256 contiguous bytes of every channel row
#define PK_CH 128     // channels per block (the grid's z also splits the descriptor): 32 KB tile, 6 blocks per SM
struct PackArgs {
  const float* src0; const float* src1; const float* scale; int Dch, Nc, Nc_pad;
  __nv_bfloat16* hi0; __nv_bfloat16* lo0; __nv_bfloat16* hi1; __nv_bfloat16* lo1;
};
// (bx, by, bz) = block coordinates in a (Nc_pad / PK_CELLS, B, tensors x channel blocks) grid; tile: PK_CH x (PK_CELLS + 1) floats
__device__ __forceinline__ void desc_pack_block(const PackArgs& A, int bx, int by, int bz, float (*tile)[PK_CELLS + 1]) {
  const float* __restrict__ src0 = A.src0; const float* __restrict__ src1 = A.src1; const float* __restrict__ scale = A.scale;
  const int Dch = A.Dch, Nc = A.Nc, Nc_pad = A.Nc_pad;
  __nv_bfloat16* __restrict__ hi0 = A.hi0; __nv_bfloat16* __restrict__ lo0 = A.lo0;
  __nv_bfloat16* __restrict__ hi1 = A.hi1; __nv_bfloat16* __restrict__ lo1 = A.lo1;
  // blockIdx.z = (tensor, channel block)
  const int nchb = (Dch + PK_CH - 1) / PK_CH;
  const int which = blockIdx.z / nchb, d0 = (blockIdx.z - which * nchb) * PK_CH;
  const float* __restrict__ src = which ? src1 : src0;
  __nv_bfloat16* __restrict__ hi = which ? hi1 : hi0;
  __nv_bfloat16* __restrict__ lo = which ? lo1 : lo0;
  const int b = by;
  const int c0 = bx * PK_CELLS;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // ---- phase 1: warp = one channel row at a time, lanes = cells (lane, lane + 32); 8 rows = 16 loads in flight per thread
  const int ca = c0 + lane, cb = ca + 32;
  float sa = 1.f, sb = 1.f;
  if (scale) {
    if (ca < Nc) sa = scale[(size_t)b * Nc_pad + ca];
    if (cb < Nc) sb = scale[(size_t)b * Nc_pad + cb];
  }
#pragma unroll 1
  for (int i0 = 0; i0 < PK_CH / 8; i0 += 8) {
    float va[8], vb[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int d = d0 + w + 8 * (i0 + u);
      const float* row = src + ((size_t)b * Dch + d) * Nc;
      va[u] = (d < Dch && ca < Nc) ? __ldg(row + ca) : 0.f;
      vb[u] = (d < Dch && cb < Nc) ? __ldg(row + cb) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int dl = w + 8 * (i0 + u);
      tile[dl][lane] = va[u] * sa;
      tile[dl][lane + 32] = vb[u] * sb;
    }
  }
  __syncthreads();
  // ---- phase 2: warp = one cell at a time, lane = channel pairs (2 lane, 2 lane + 1) + 64 j: one packed conversion
  // (cvt.rn.bf16x2.f32) per pair for hi, one for lo, and 4-byte stores: 128 contiguous bytes per warp store.
  // (The two scalar LDS per pair are 2-way bank conflicted; the kernel is bound by issued instructions, not by LDS.)
#pragma unroll 2
  for (int cc = w; cc < PK_CELLS; cc += 8) {
    const size_t o = ((size_t)b * Nc_pad + c0 + cc) * Dch + d0;
#pragma unroll
    for (int j = 0; j < PK_CH / 64; ++j) {
      const int d = 2 * lane + 64 * j;
      const float v0 = tile[d][cc], v1 = tile[d + 1][cc];
      uint32_t h2, l2;
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h2) : "f"(v1), "f"(v0));  // low half = v0
      const float r0 = v0 - __uint_as_float(h2 << 16), r1 = v1 - __uint_as_float(h2 & 0xffff0000u);
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(l2) : "f"(r1), "f"(r0));
      if (d0 + d < Dch) {
        *reinterpret_cast<uint32_t*>(hi + o + d) = h2;
        if (lo) *reinterpret_cast<uint32_t*>(lo + o + d) = l2;
      }
    }
  }
}

__global__ void __launch_bounds__(256) desc_pack_kernel(const __grid_constant__ PackArgs A) {
  __shared__ float tile[PK_CH][PK_CELLS + 1];
  desc_pack_block(A, blockIdx.x, blockIdx.y, blockIdx.z, tile);
}

// Forward prologue of the descriptor loss: the operand pack (z < npack) and the geometry kernel (z == npack; only its first
// Nc_pad / 256 x-blocks exist) do not depend on each other -- one launch instead of two, the light geometry blocks fill in
// next to the streaming pack blocks.
__global__ void __launch_bounds__(256)
desc_pack_geometry_kernel(const __grid_constant__ PackArgs P, const __grid_constant__ GeomArgs G, int npack, int ggx) {
  __shared__ __align__(16) float tile[PK_CH][PK_CELLS + 1];
  if ((int)blockIdx.z < npack) {
    desc_pack_block(P, blockIdx.x, blockIdx.y, blockIdx.z, tile);
  } else if ((int)blockIdx.x < ggx) {
    desc_geometry_block(G, blockIdx.x, blockIdx.y, ggx, reinterpret_cast<double*>(&tile[0][0]));
  }
}

// One tensor; `scale` (optional) multiplies its cells.
extern "C" int ssp_desc_pack(const float* src, const float* scale, int B, int Dch, int Nc, void* hi, void* lo,
                             void* stream) {
  SSP_REQUIRE(src && hi, "ssp_desc_pack: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && Dch > 0 && Dch % 2 == 0 && Nc > 0, "ssp_desc_pack: bad sizes (Dch must be even)");
  int Nc_pad = desc_nc_pad(Nc);
  const int nchb = (Dch + PK_CH - 1) / PK_CH;
  SSP_REQUIRE(nchb <= 65535, "ssp_desc_pack: descriptor dim %d too large", Dch);
  dim3 grid(Nc_pad / PK_CELLS, B, nchb);
  PackArgs A = {src, nullptr, scale, Dch, Nc, Nc_pad, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, nullptr, nullptr};
  desc_pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
  SSP_CUDA_CHECK_LAUNCH("desc_pack_kernel");
  return SSP_OK;
}

// two ssp_desc_pack calls (no scale) and the descriptor-loss geometry as ONE launch.  hi0 == hi1 == NULL: the geometry
// alone (src*, lo* and Dch unused), for the fp32 engine, which reads no planes.
// mvbits (optional): [B, Nc_pad/32] words of mask_valid != 0 in DESC_BITPOS order for the "fold" mode of the tensor-core
// engine; requesting them also makes a non-binary mask poison the normaliser with NaN.
// mask2d (optional, used when mask_valid is NULL): the pixel-resolution mask [B,1,8Hc,8Wc] the cell mask is the product of
// (getMasks fused in; cell must be 8).
extern "C" int ssp_desc_pack2_geometry(const float* src0, const float* src1, int B, int Dch, int Hc, int Wc, void* hi0, void* lo0,
                                       void* hi1, void* lo1, const float* Hm, const float* mask_valid, const float* mask2d,
                                       int cell, float* wpts, float* mv_pad, double* mv_part, uint32_t* mvbits, void* stream) {
  const bool pack = hi0 || hi1;
  SSP_REQUIRE((!pack || (src0 && src1 && hi0 && hi1)) && Hm && wpts && mv_pad && mv_part, "ssp_desc_pack2_geometry: null pointer");
  SSP_REQUIRE(B > 0 && B <= 65535 && (!pack || (Dch > 0 && Dch % 2 == 0)) && Hc > 0 && Wc > 0 && cell > 0,
              "ssp_desc_pack2_geometry: bad sizes");
  SSP_REQUIRE(!mask2d || mask_valid || (cell == 8 && ((uintptr_t)mask2d & 15) == 0),
              "ssp_desc_pack2_geometry: the fused pixel mask needs cell_size 8 and a 16-byte aligned mask");
  const int Nc = Hc * Wc, Nc_pad = desc_nc_pad(Nc);
  GeomArgs G = {Hm, mask_valid, mask2d, B, Hc, Wc, cell, Nc_pad, reinterpret_cast<float2*>(wpts), mv_pad, mv_part, mvbits};
  if (!pack) {
    // not desc_pack_geometry_kernel with npack = 0: its 33 KB pack tile made the geometry 7.4 instead of 5.3 us and the
    // positive-pair kernel after it 52.3 instead of 51.0 us (fp32 engine, B = 32 of 30 x 40 cells, NVIDIA B200 at 1000 W)
    desc_geometry_kernel<<<dim3(Nc_pad / GEOM_THREADS, B), GEOM_THREADS, 0, (cudaStream_t)stream>>>(G);
    SSP_CUDA_CHECK_LAUNCH("desc_geometry_kernel");
    return SSP_OK;
  }
  const int npack = 2 * ((Dch + PK_CH - 1) / PK_CH);
  SSP_REQUIRE(npack + 1 <= 65535, "ssp_desc_pack2_geometry: descriptor dim %d too large", Dch);
  PackArgs P = {src0, src1, nullptr, Dch, Nc, Nc_pad, (__nv_bfloat16*)hi0, (__nv_bfloat16*)lo0, (__nv_bfloat16*)hi1, (__nv_bfloat16*)lo1};
  dim3 grid(Nc_pad / PK_CELLS, B, npack + 1);
  desc_pack_geometry_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(P, G, npack, Nc_pad / GEOM_THREADS);
  SSP_CUDA_CHECK_LAUNCH("desc_pack_geometry_kernel");
  return SSP_OK;
}
