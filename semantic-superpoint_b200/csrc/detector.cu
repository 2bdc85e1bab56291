// Detector label / loss path and heatmap flattening.
// Reference semantics (Gabriel-SGama/Semantic-SuperPoint):
//   labels2Dto3D            utils/utils.py:408-440   (+ SpaceToDepth utils/d2s.py:27-44)
//   getMasks                Train_model_frontend_all.py:373-386
//   detector_loss (softmax) Train_model_heatmap_all.py:155-179  -> BCE over softmax probabilities
//   flattenDetection        utils/utils.py:515-560   (+ DepthToSpace utils/d2s.py:8-25)
// Layout: one thread per 8x8 cell; the 65 channel values of a cell are Nc floats apart (NCHW), so a
// warp reads 32 consecutive cells of one channel = one 128 B line; the 8x8 pixel block of a cell is
// 8 rows of 32 B, read/written as 2 x float4 per row.  All kernels are HBM-bound.
#include "common.cuh"
#include "desc_pos_coef.cuh"

#define CELL 8
#define NCH 65

// ----------------------------------------------------------------------------------------------
// labels2Dto3D: pixel-unshuffle(8) (+ dustbin + normalisation)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_cell(const float* __restrict__ img, int W, int y0, int x0, float (&v)[64]) {
#pragma unroll
  for (int dy = 0; dy < CELL; ++dy) {
    const float4* r = reinterpret_cast<const float4*>(img + (size_t)(y0 + dy) * W + x0);
    float4 a = __ldg(r), b = __ldg(r + 1);
    v[dy * 8 + 0] = a.x; v[dy * 8 + 1] = a.y; v[dy * 8 + 2] = a.z; v[dy * 8 + 3] = a.w;
    v[dy * 8 + 4] = b.x; v[dy * 8 + 5] = b.y; v[dy * 8 + 6] = b.z; v[dy * 8 + 7] = b.w;
  }
}

// dustbin + normaliser exactly as the reference: d = 1 - sum; d < 1 -> 0; divide all 65 by their sum
__device__ __forceinline__ void dustbin_norm(float (&v)[64], float& dust) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 64; ++c) s += v[c];
  dust = 1.f - s;
  if (dust < 1.f) dust = 0.f;
  float dn = s + dust;
#pragma unroll
  for (int c = 0; c < 64; ++c) v[c] = v[c] / dn;
  dust = dust / dn;
}

__global__ void __launch_bounds__(128)
labels2d_to_3d_kernel(const float* __restrict__ labels, int B, int H, int W, int add_dustbin,
                      float* __restrict__ out) {
  int Hc = H / CELL, Wc = W / CELL, Nc = Hc * Wc;
  int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= B * Nc) return;
  int b = cell / Nc, ij = cell % Nc;
  int k = ij / Wc, l = ij % Wc;
  float v[64];
  load_cell(labels + (size_t)b * H * W, W, k * CELL, l * CELL, v);
  int nch = add_dustbin ? 65 : 64;
  float dust = 0.f;
  if (add_dustbin) dustbin_norm(v, dust);
  float* o = out + (size_t)b * nch * Nc + ij;
#pragma unroll
  for (int c = 0; c < 64; ++c) o[(size_t)c * Nc] = v[c];
  if (add_dustbin) o[(size_t)64 * Nc] = dust;
}

extern "C" int ssp_labels2d_to_3d(const float* labels, int B, int H, int W, int add_dustbin, float* out,
                                  void* stream) {
  SSP_REQUIRE(labels && out, "ssp_labels2d_to_3d: null pointer");
  SSP_REQUIRE(B > 0 && H >= CELL && W >= CELL && H % CELL == 0 && W % CELL == 0,
              "ssp_labels2d_to_3d: H=%d W=%d must be positive multiples of 8 (B=%d)", H, W, B);
  int cells = B * (H / CELL) * (W / CELL);
  labels2d_to_3d_kernel<<<ssp_ceil_div(cells, 128), 128, 0, (cudaStream_t)stream>>>(labels, B, H, W, add_dustbin, out);
  SSP_CUDA_CHECK_LAUNCH("labels2d_to_3d_kernel");
  return SSP_OK;
}

// getMasks: product of the 64 sub-pixels of every cell
__global__ void __launch_bounds__(128)
cell_mask_kernel(const float* __restrict__ mask2d, int B, int H, int W, float* __restrict__ out) {
  int Hc = H / CELL, Wc = W / CELL, Nc = Hc * Wc;
  int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= B * Nc) return;
  int b = cell / Nc, ij = cell % Nc;
  float v[64];
  load_cell(mask2d + (size_t)b * H * W, W, (ij / Wc) * CELL, (ij % Wc) * CELL, v);
  float p = v[0];
#pragma unroll
  for (int c = 1; c < 64; ++c) p *= v[c];
  out[cell] = p;
}

extern "C" int ssp_cell_mask(const float* mask2d, int B, int H, int W, float* out, void* stream) {
  SSP_REQUIRE(mask2d && out, "ssp_cell_mask: null pointer");
  SSP_REQUIRE(B > 0 && H >= CELL && W >= CELL && H % CELL == 0 && W % CELL == 0,
              "ssp_cell_mask: H=%d W=%d must be positive multiples of 8 (B=%d)", H, W, B);
  int cells = B * (H / CELL) * (W / CELL);
  cell_mask_kernel<<<ssp_ceil_div(cells, 128), 128, 0, (cudaStream_t)stream>>>(mask2d, B, H, W, out);
  SSP_CUDA_CHECK_LAUNCH("cell_mask_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// detector loss: sum_cells mask * sum_c BCE(softmax(semi)_c, target_c) / (sum mask + 1e-5)
// Block = 32 cells x 4 channel groups (warp g owns channels 16g..16g+15, warp 3 also the dustbin 64), i.e.
// 4 threads per cell: 4x the memory-level parallelism and a quarter of the registers of a thread-per-cell
// layout.  In the fused-2D variant warp g reads pixel rows 2g, 2g+1 of every 8x8 cell (channel = dy*8+dx).
// ----------------------------------------------------------------------------------------------
#define DET_CELLS 32
#define DET_GROUPS 4
#define DET_CPG 16  // channels per group

// MUFU-level transcendental helpers.  The loss needs 65 exponentials and 130 logarithms per cell; with libm expf /
// logf / IEEE divisions the kernels were instruction-bound (1700 SASS instructions per thread, ncu issue-active 63 %,
// 29 % of the HBM roofline).  ex2.approx / lg2.approx are accurate to 2 ulp, far inside the 1e-4 parity tolerance.
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
#define DET_LOG2E 1.4426950408889634f
#define DET_LN2 0.6931471805599453f

struct DetShared {
  float red[3][DET_GROUPS][DET_CELLS];
};

// combine one value per channel group into the per-cell total (fixed order 0..3), all threads get it
template <typename Op>
__device__ __forceinline__ float det_combine(DetShared& sh, float v, int lane, int grp, Op op) {
  __syncthreads();
  sh.red[0][grp][lane] = v;
  __syncthreads();
  return op(op(sh.red[0][0][lane], sh.red[0][1][lane]), op(sh.red[0][2][lane], sh.red[0][3][lane]));
}

// Everything a thread needs, loaded up front so that all global loads of a cell are in flight together:
// 16 (+1) logits, 16 (+1) target values (raw 2-D labels when FUSED2D) and the mask (partial product when FUSED2D).
template <int FUSED2D>
__device__ __forceinline__ void det_load(const float* __restrict__ semi_cell, const float* __restrict__ target,
                                         const float* __restrict__ mask, int b, int ij, int cell, int Hc, int Wc, bool valid,
                                         int grp, float (&x)[DET_CPG], float& xd, float (&t)[DET_CPG], float& td, float& mk) {
  const int Nc = Hc * Wc;  // 32-bit channel offsets: one IMAD.WIDE per load instead of a 64-bit multiply chain
  const float* __restrict__ sp = semi_cell + (size_t)(grp * DET_CPG) * Nc;
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) x[c] = valid ? __ldg(sp + c * Nc) : 0.f;
  xd = (valid && grp == 3) ? __ldg(sp + DET_CPG * Nc) : -INFINITY;
  td = 0.f;
  if (FUSED2D) {
    int H = Hc * CELL, W = Wc * CELL;
    int y0 = (ij / Wc) * CELL + 2 * grp, x0 = (ij % Wc) * CELL;
    mk = 1.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      float4 a = make_float4(0, 0, 0, 0), c4 = a, ma = make_float4(1, 1, 1, 1), mb = ma;
      if (valid) {
        const float4* r = reinterpret_cast<const float4*>(target + ((size_t)b * H + y0 + dy) * W + x0);
        const float4* q = reinterpret_cast<const float4*>(mask + ((size_t)b * H + y0 + dy) * W + x0);
        a = __ldg(r); c4 = __ldg(r + 1); ma = __ldg(q); mb = __ldg(q + 1);
      }
      t[dy * 8 + 0] = a.x; t[dy * 8 + 1] = a.y; t[dy * 8 + 2] = a.z; t[dy * 8 + 3] = a.w;
      t[dy * 8 + 4] = c4.x; t[dy * 8 + 5] = c4.y; t[dy * 8 + 6] = c4.z; t[dy * 8 + 7] = c4.w;
      mk *= ma.x * ma.y * ma.z * ma.w * mb.x * mb.y * mb.z * mb.w;
    }
  } else {
    mk = valid ? __ldg(mask + cell) : 0.f;
    const float* __restrict__ tp = target + (size_t)b * NCH * Nc + ij + (size_t)(grp * DET_CPG) * Nc;
#pragma unroll
    for (int c = 0; c < DET_CPG; ++c) t[c] = valid ? __ldg(tp + c * Nc) : 0.f;
    if (grp == 3) td = valid ? __ldg(tp + DET_CPG * Nc) : 0.f;
  }
}

// Softmax of the cell in the log2 domain, normalised targets and the cell mask: two barrier rounds (max; then
// exp-sum, label-sum and mask-product together).  On return
//   v[c]  = (x_c - max) * log2(e)      (pd likewise for the dustbin channel of group 3)
//   e[c]  = 2^v[c]                     (ed)
//   inv_se = 1 / sum_c e_c,  lnse = ln(sum_c e_c)   ->  p_c = e_c * inv_se,  ln p_c = v_c * ln2 - lnse
//   t[c]  = target / (sum + dustbin)   (FUSED2D; already normalised otherwise),  mk = cell mask
template <int FUSED2D>
__device__ __forceinline__ void det_prepare(DetShared& sh, int lane, int grp, float (&v)[DET_CPG], float& vd,
                                            float (&e)[DET_CPG], float& ed, float (&t)[DET_CPG], float& td, float& mk,
                                            float& inv_se, float& lnse) {
  float m = vd;  // -inf unless this thread owns the dustbin channel
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) m = fmaxf(m, v[c]);
  m = det_combine(sh, m, lane, grp, [](float a, float b) { return fmaxf(a, b); });
  const float ms = m * DET_LOG2E;
  float se = 0.f, ls = 0.f;
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) {
    v[c] = fmaf(v[c], DET_LOG2E, -ms);
    e[c] = fast_ex2(v[c]);
    se += e[c];
    ls += t[c];
  }
  ed = 0.f;
  if (grp == 3) {
    vd = fmaf(vd, DET_LOG2E, -ms);
    ed = fast_ex2(vd);
    se += ed;
  }
  __syncthreads();
  sh.red[0][grp][lane] = se;
  sh.red[1][grp][lane] = ls;
  sh.red[2][grp][lane] = mk;
  __syncthreads();
  se = (sh.red[0][0][lane] + sh.red[0][1][lane]) + (sh.red[0][2][lane] + sh.red[0][3][lane]);
  inv_se = 1.f / se;
  lnse = fast_lg2(se) * DET_LN2;
  if (FUSED2D) {
    float s = (sh.red[1][0][lane] + sh.red[1][1][lane]) + (sh.red[1][2][lane] + sh.red[1][3][lane]);
    mk = (sh.red[2][0][lane] * sh.red[2][1][lane]) * (sh.red[2][2][lane] * sh.red[2][3][lane]);
    // dustbin: d = 1 - sum; d < 1 -> 0; all 65 channels divided by their sum   [utils/utils.py:431-439]
    float dust = 1.f - s;
    if (dust < 1.f) dust = 0.f;
    float dn = s + dust;
    float inv_dn = 1.f / dn;
    if (dn != 1.f) {  // block-uniform in the common case (binary labels: empty cell or one keypoint)
#pragma unroll
      for (int c = 0; c < DET_CPG; ++c) t[c] = t[c] * inv_dn;
    }
    td = dust * inv_dn;
  }
}

// BCE of one channel given e = 2^v: -(t ln p + (1-t) ln(1-p)), both logarithms clamped at -100 like nn.BCELoss.
// ln p is taken from the logits (v ln2 - ln se), so only ln(1-p) costs a MUFU.
__device__ __forceinline__ float bce_term(float v, float e, float t, float inv_se, float lnse) {
  float p = e * inv_se;
  float lp = fmaxf(fmaf(v, DET_LN2, -lnse), -100.f);
  float lq = fmaxf(fast_lg2(1.f - p) * DET_LN2, -100.f);
  return fmaf(t, lq - lp, -lq);
}

// One launch serves up to two independent losses (image and warped image of a training pair): blockIdx.y selects
// the problem.  Halves the number of launches / latency chains of the loss step.
struct DetProblem {
  const float* semi;
  const float* target;
  const float* mask;
  double* partials;
  unsigned int* counter;
  float* out;          // forward: out3; backward: dsemi
  float* cellmask;     // forward only, optional: per-cell mask product [B,Hc,Wc] (= getMasks), else nullptr
  const float* fwd_out;  // backward only
  const float* gout;     // backward only
};
struct DetProblems {
  DetProblem p[2];
};

// FUSED2D = 0: target [B,65,Hc,Wc] and mask [B,Hc,Wc] are given (reference call signature).
// FUSED2D = 1: target/mask are built on the fly from labels_2D / mask_2D [B,1,H,W].
template <int FUSED2D>
__global__ void __launch_bounds__(DET_CELLS * DET_GROUPS)
detector_loss_fwd_kernel(const __grid_constant__ DetProblems probs, int B, int Hc, int Wc) {
  const DetProblem& pr = probs.p[blockIdx.y];
  const float* __restrict__ semi = pr.semi;
  const float* __restrict__ target = pr.target;
  const float* __restrict__ mask = pr.mask;
  double* __restrict__ partials = pr.partials;
  __shared__ DetShared sh;
  int Nc = Hc * Wc;
  int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  int cell = blockIdx.x * DET_CELLS + lane;
  bool valid = cell < B * Nc;
  int b = valid ? cell / Nc : 0, ij = valid ? cell % Nc : 0;
  float v[DET_CPG], e[DET_CPG], t[DET_CPG], vd, ed, td, mk, inv_se, lnse;
  det_load<FUSED2D>(semi + (size_t)b * NCH * Nc + ij, target, mask, b, ij, cell, Hc, Wc, valid, grp, v, vd, t, td, mk);
  det_prepare<FUSED2D>(sh, lane, grp, v, vd, e, ed, t, td, mk, inv_se, lnse);
  float bce = 0.f;
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) bce += bce_term(v[c], e[c], t[c], inv_se, lnse);
  if (grp == 3) bce += bce_term(vd, ed, td, inv_se, lnse);
  bce = det_combine(sh, bce, lane, grp, [](float a, float b) { return a + b; });
  // per-block partials (32 cells, summed in fp32 by warp 0); a one-block-per-problem finalize kernel adds them in
  // double, in index order: deterministic, and no same-address atomics.
  if (grp == 0) {
    float num = valid ? bce * mk : 0.f, den = valid ? mk : 0.f;
    if (valid && pr.cellmask) pr.cellmask[cell] = mk;
    num = warp_sum(num);
    den = warp_sum(den);
    if (lane == 0) {
      partials[2 * (size_t)blockIdx.x] = (double)num;
      partials[2 * (size_t)blockIdx.x + 1] = (double)den;
    }
  }
}

__global__ void __launch_bounds__(256)
detector_loss_finalize_kernel(const __grid_constant__ DetProblems probs, int nblk) {
  const DetProblem& pr = probs.p[blockIdx.x];
  __shared__ double shd[32];
  double a = 0.0, c = 0.0;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) {
    a += pr.partials[2 * (size_t)i];
    c += pr.partials[2 * (size_t)i + 1];
  }
  a = block_sum_d(a, shd);
  c = block_sum_d(c, shd);
  if (threadIdx.x == 0) {
    float num = (float)a;
    float den = (float)c + 1e-5f;
    pr.out[0] = num / den;  // loss
    pr.out[1] = num;
    pr.out[2] = den;
  }
}

// d semi = gout * mask/den * softmax_bwd( (p - t) / max(p (1-p), 1e-12) )
// (the body is a device function over the block index so that the fused step's backward prologue can run it as some of the
// blocks of a launch whose other blocks are the descriptor backward's coefficient / transpose blocks)
template <int FUSED2D>
__device__ __forceinline__ void det_bwd_block(const DetProblem& pr, int B, int Hc, int Wc, int bx, DetShared& sh) {
  const float* __restrict__ semi = pr.semi;
  const float* __restrict__ target = pr.target;
  const float* __restrict__ mask = pr.mask;
  const float* __restrict__ fwd_out = pr.fwd_out;
  const float* __restrict__ gout = pr.gout;
  float* __restrict__ dsemi = pr.out;
  int Nc = Hc * Wc;
  int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  int cell = bx * DET_CELLS + lane;
  bool valid = cell < B * Nc;
  int b = valid ? cell / Nc : 0, ij = valid ? cell % Nc : 0;
  float v[DET_CPG], e[DET_CPG], t[DET_CPG], vd, ed, td, mk, inv_se, lnse;
  det_load<FUSED2D>(semi + (size_t)b * NCH * Nc + ij, target, mask, b, ij, cell, Hc, Wc, valid, grp, v, vd, t, td, mk);
  det_prepare<FUSED2D>(sh, lane, grp, v, vd, e, ed, t, td, mk, inv_se, lnse);
  // g_c = dBCE/dp_c = (p - t) / max(p (1 - p), 1e-12);  d semi_c = scale * p_c * (g_c - sum_k p_k g_k)
  float dot = 0.f, gd = 0.f;
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) {
    float p = e[c] * inv_se;
    float g = (p - t[c]) * fast_rcp(fmaxf((1.f - p) * p, 1e-12f));
    e[c] = p;
    t[c] = g;
    dot = fmaf(p, g, dot);
  }
  if (grp == 3) {
    float p = ed * inv_se;
    gd = (p - td) * fast_rcp(fmaxf((1.f - p) * p, 1e-12f));
    ed = p;
    dot = fmaf(p, gd, dot);
  }
  dot = det_combine(sh, dot, lane, grp, [](float a, float b) { return a + b; });
  if (!valid) return;
  const float scale = __ldg(gout) * mk / __ldg(fwd_out + 2);
  float* __restrict__ o = dsemi + (size_t)b * NCH * Nc + ij + (size_t)(grp * DET_CPG) * Nc;
#pragma unroll
  for (int c = 0; c < DET_CPG; ++c) o[c * Nc] = (e[c] * scale) * (t[c] - dot);
  if (grp == 3) o[DET_CPG * Nc] = (ed * scale) * (gd - dot);
}

template <int FUSED2D>
__global__ void __launch_bounds__(DET_CELLS * DET_GROUPS)
detector_loss_bwd_kernel(const __grid_constant__ DetProblems probs, int B, int Hc, int Wc) {
  __shared__ DetShared sh;
  det_bwd_block<FUSED2D>(probs.p[blockIdx.y], B, Hc, Wc, blockIdx.x, sh);
}

// Backward prologue of the fused loss step: ONE launch whose first blocks are the descriptor backward's coefficient /
// alpha / bit-transpose blocks (chains of dependent gathers and small streaming transposes) and whose remaining blocks are
// the detector-loss backward of both images (HBM-bound).  As separate kernels they run back to back, each filling the GPU
// with its own kind of stall; as blocks of one grid they share the SMs.  1-D grid: [pgx * pgy * pgz descriptor blocks |
// ndet blocks of problem 0 | ndet blocks of problem 1].
template <int FUSED2D>
__global__ void __launch_bounds__(DET_CELLS * DET_GROUPS, 8)  // 64 registers: the detector blocks keep their stand-alone occupancy
step_bwd_prologue_kernel(const __grid_constant__ DetProblems probs, const __grid_constant__ PosCoefArgs pc, int B, int Hc, int Wc,
                         int ndet, int pgx, int pgy, int pgz) {
  __shared__ DetShared sh;
  int id = blockIdx.x;
  const int npc = pgx * pgy * pgz;
  if (id < npc) {
    const int bz = id / (pgx * pgy), r = id - bz * (pgx * pgy);
    const int by = r / pgx, bx = r - by * pgx;
    desc_pos_coef_block(pc, bx, by, bz, pgx);
    return;
  }
  id -= npc;
  const int prob = id / ndet;
  det_bwd_block<FUSED2D>(probs.p[prob], B, Hc, Wc, id - prob * ndet, sh);
}

extern "C" size_t ssp_detector_loss_ws_bytes(int B, int Hc, int Wc) {
  size_t nblk = (size_t)ssp_ceil_div(B * Hc * Wc, DET_CELLS);
  return 16 + nblk * 2 * sizeof(double);
}

static int det_check(const char* who, const float* semi, const float* target, const float* mask, int B, int Hc, int Wc,
                     int fused2d) {
  SSP_REQUIRE(semi && target && mask, "%s: null pointer", who);
  SSP_REQUIRE(B > 0 && Hc > 0 && Wc > 0, "%s: bad sizes B=%d Hc=%d Wc=%d", who, B, Hc, Wc);
  if (fused2d)
    SSP_REQUIRE((((uintptr_t)target | (uintptr_t)mask) & 15) == 0, "%s: 2-D label/mask pointers must be 16-byte aligned", who);
  return SSP_OK;
}

// Forward of one (semi1 == NULL) or two losses in one launch.  ws holds one region of ssp_detector_loss_ws_bytes per
// problem.  cellmask1 (optional) receives the per-cell mask product of problem 1 (the descriptor loss's mask_valid).
extern "C" int ssp_detector_loss_fwd_pair(const float* semi0, const float* target0, const float* mask0,
                                          const float* semi1, const float* target1, const float* mask1, int B, int Hc,
                                          int Wc, int fused2d, float* out3_0, float* out3_1, float* cellmask1, void* ws,
                                          size_t ws_bytes, void* stream) {
  int rc;
  if ((rc = det_check("ssp_detector_loss_fwd_pair", semi0, target0, mask0, B, Hc, Wc, fused2d))) return rc;
  int np = semi1 ? 2 : 1;
  if (np == 2 && (rc = det_check("ssp_detector_loss_fwd_pair", semi1, target1, mask1, B, Hc, Wc, fused2d))) return rc;
  SSP_REQUIRE(out3_0 && ws && (np == 1 || out3_1), "ssp_detector_loss_fwd_pair: null pointer");
  size_t per = (ssp_detector_loss_ws_bytes(B, Hc, Wc) + 15) / 16 * 16;
  SSP_REQUIRE(ws_bytes >= per * np, "ssp_detector_loss_fwd_pair: workspace too small");
  SSP_REQUIRE(((uintptr_t)ws & 15) == 0, "ssp_detector_loss_fwd_pair: workspace must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  DetProblems pb = {};
  for (int i = 0; i < np; ++i) {
    char* w = (char*)ws + per * i;
    pb.p[i].semi = i ? semi1 : semi0;
    pb.p[i].target = i ? target1 : target0;
    pb.p[i].mask = i ? mask1 : mask0;
    pb.p[i].counter = (unsigned int*)w;
    pb.p[i].partials = (double*)(w + 16);
    pb.p[i].out = i ? out3_1 : out3_0;
    pb.p[i].cellmask = i ? cellmask1 : nullptr;
  }
  dim3 grid(ssp_ceil_div(B * Hc * Wc, DET_CELLS), np);
  if (fused2d)
    detector_loss_fwd_kernel<1><<<grid, 128, 0, st>>>(pb, B, Hc, Wc);
  else
    detector_loss_fwd_kernel<0><<<grid, 128, 0, st>>>(pb, B, Hc, Wc);
  SSP_CUDA_CHECK_LAUNCH("detector_loss_fwd_kernel");
  detector_loss_finalize_kernel<<<np, 256, 0, st>>>(pb, (int)grid.x);
  SSP_CUDA_CHECK_LAUNCH("detector_loss_finalize_kernel");
  return SSP_OK;
}

extern "C" int ssp_detector_loss_bwd_pair(const float* semi0, const float* target0, const float* mask0,
                                          const float* semi1, const float* target1, const float* mask1, int B, int Hc,
                                          int Wc, int fused2d, const float* fwd0, const float* fwd1, const float* gout0,
                                          const float* gout1, float* dsemi0, float* dsemi1, void* stream) {
  int rc;
  if ((rc = det_check("ssp_detector_loss_bwd_pair", semi0, target0, mask0, B, Hc, Wc, fused2d))) return rc;
  int np = semi1 ? 2 : 1;
  if (np == 2 && (rc = det_check("ssp_detector_loss_bwd_pair", semi1, target1, mask1, B, Hc, Wc, fused2d))) return rc;
  SSP_REQUIRE(fwd0 && gout0 && dsemi0 && (np == 1 || (fwd1 && gout1 && dsemi1)), "ssp_detector_loss_bwd_pair: null pointer");
  DetProblems pb = {};
  for (int i = 0; i < np; ++i) {
    pb.p[i].semi = i ? semi1 : semi0;
    pb.p[i].target = i ? target1 : target0;
    pb.p[i].mask = i ? mask1 : mask0;
    pb.p[i].out = i ? dsemi1 : dsemi0;
    pb.p[i].fwd_out = i ? fwd1 : fwd0;
    pb.p[i].gout = i ? gout1 : gout0;
  }
  dim3 grid(ssp_ceil_div(B * Hc * Wc, DET_CELLS), np);
  cudaStream_t st = (cudaStream_t)stream;
  if (fused2d)
    detector_loss_bwd_kernel<1><<<grid, 128, 0, st>>>(pb, B, Hc, Wc);
  else
    detector_loss_bwd_kernel<0><<<grid, 128, 0, st>>>(pb, B, Hc, Wc);
  SSP_CUDA_CHECK_LAUNCH("detector_loss_bwd_kernel");
  return SSP_OK;
}

// Fused-step backward prologue: ssp_detector_loss_bwd_pair (fused2d = 1, both images) and ssp_desc_pos_coef (with alpha / srow
// / bitsC outputs) as ONE launch.  Arguments = those two calls'.
extern "C" int ssp_step_bwd_prologue(const float* semi0, const float* labels0, const float* mask0, const float* semi1,
                                     const float* labels1, const float* mask1, int B, int Hc, int Wc, const float* fwd0,
                                     const float* fwd1, const float* gout, float* dsemi0, float* dsemi1,
                                     const int* rowcol, const float* rowdot, const int* colcnt, const int* colrow,
                                     const float* coldot, const uint32_t* bitsR, const float* mv_pad, const float* g3,
                                     float gscale, int gmode, const float* out8, float lamda, float mpos, float* rowcoef,
                                     int* colrow_sorted, float* colcoef, float* alpha_out, float* srow_out,
                                     uint32_t* bitsC_out, void* stream) {
  int rc;
  if ((rc = det_check("ssp_step_bwd_prologue", semi0, labels0, mask0, B, Hc, Wc, 1))) return rc;
  if ((rc = det_check("ssp_step_bwd_prologue", semi1, labels1, mask1, B, Hc, Wc, 1))) return rc;
  SSP_REQUIRE(fwd0 && fwd1 && gout && dsemi0 && dsemi1, "ssp_step_bwd_prologue: null pointer (detector side)");
  SSP_REQUIRE(rowcol && rowdot && colcnt && colrow && coldot && bitsR && mv_pad && g3 && out8 && rowcoef && colrow_sorted && colcoef,
              "ssp_step_bwd_prologue: null pointer (descriptor side)");
  SSP_REQUIRE(B <= 65535 && (gmode == 0 || gmode == 1), "ssp_step_bwd_prologue: bad sizes");
  const int Nc = Hc * Wc, Nc_pad = desc_nc_pad(Nc);
  DetProblems pb = {};
  for (int i = 0; i < 2; ++i) {
    pb.p[i].semi = i ? semi1 : semi0;
    pb.p[i].target = i ? labels1 : labels0;
    pb.p[i].mask = i ? mask1 : mask0;
    pb.p[i].out = i ? dsemi1 : dsemi0;
    pb.p[i].fwd_out = i ? fwd1 : fwd0;
    pb.p[i].gout = gout;
  }
  PosCoefArgs A = {rowcol, rowdot, colcnt, colrow, coldot, bitsR, mv_pad, g3, gscale, gmode, out8, Nc_pad, lamda, mpos,
                   rowcoef, colrow_sorted, colcoef, alpha_out, srow_out, bitsC_out, (Nc + 31) / 32};
  const int ndet = ssp_ceil_div(B * Nc, DET_CELLS), pgx = Nc_pad / 128, pgy = B, pgz = bitsC_out ? 6 : 2;
  const long long nblk = (long long)pgx * pgy * pgz + 2ll * ndet;
  SSP_REQUIRE(nblk < 0x7fffffffll, "ssp_step_bwd_prologue: grid too large");
  step_bwd_prologue_kernel<1><<<(unsigned)nblk, 128, 0, (cudaStream_t)stream>>>(pb, A, B, Hc, Wc, ndet, pgx, pgy, pgz);
  SSP_CUDA_CHECK_LAUNCH("step_bwd_prologue_kernel");
  return SSP_OK;
}

// ----------------------------------------------------------------------------------------------
// flattenDetection: softmax(65) -> drop dustbin -> pixel-shuffle(8)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void softmax65(const float* __restrict__ semi_cell, size_t Nc, float (&p)[NCH]) {
  float m = -INFINITY;
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    p[c] = __ldg(semi_cell + (size_t)c * Nc);
    m = fmaxf(m, p[c]);
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    p[c] = expf(p[c] - m);
    s += p[c];
  }
#pragma unroll
  for (int c = 0; c < NCH; ++c) p[c] = p[c] / s;
}

__global__ void __launch_bounds__(128)
flatten_detection_kernel(const float* __restrict__ semi, int N, int Hc, int Wc, float* __restrict__ heat) {
  int Nc = Hc * Wc;
  int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= N * Nc) return;
  int b = cell / Nc, ij = cell % Nc;
  int k = ij / Wc, l = ij % Wc;
  float p[NCH];
  softmax65(semi + (size_t)b * NCH * Nc + ij, Nc, p);
  int W = Wc * CELL;
  float* o = heat + (size_t)b * Nc * 64 + (size_t)(k * CELL) * W + l * CELL;
#pragma unroll
  for (int dy = 0; dy < CELL; ++dy) {
    float4* r = reinterpret_cast<float4*>(o + (size_t)dy * W);
    r[0] = make_float4(p[dy * 8 + 0], p[dy * 8 + 1], p[dy * 8 + 2], p[dy * 8 + 3]);
    r[1] = make_float4(p[dy * 8 + 4], p[dy * 8 + 5], p[dy * 8 + 6], p[dy * 8 + 7]);
  }
}

// flattenDetection fused with the valid mask of the view, for the homography-adaptation aggregation (export.py:49-60 forms
// heat * mask before warping): out = heat where mask == 1, -1 where mask == 0 (heat is a softmax output, never negative, so the
// sign carries the mask and the aggregation gathers ONE array instead of two).  Any other mask value raises *flag and the
// aggregation poisons its result.
__global__ void __launch_bounds__(128)
flatten_detection_masked_kernel(const float* __restrict__ semi, const float* __restrict__ mask, int N, int Hc, int Wc,
                                float* __restrict__ heat, int* __restrict__ flag) {
  int Nc = Hc * Wc;
  int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= N * Nc) return;
  int b = cell / Nc, ij = cell % Nc;
  int k = ij / Wc, l = ij % Wc;
  float p[NCH];
  softmax65(semi + (size_t)b * NCH * Nc + ij, Nc, p);
  int W = Wc * CELL;
  const size_t off = (size_t)b * Nc * 64 + (size_t)(k * CELL) * W + l * CELL;
  bool bad = false;
#pragma unroll
  for (int dy = 0; dy < CELL; ++dy) {
    const float4* mr = reinterpret_cast<const float4*>(mask + off + (size_t)dy * W);
    const float4 m0 = __ldg(mr), m1 = __ldg(mr + 1);
    const float m[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
    float v[8];
#pragma unroll
    for (int dx = 0; dx < 8; ++dx) {
      v[dx] = m[dx] == 1.f ? p[dy * 8 + dx] : -1.f;
      bad |= !(m[dx] == 1.f || m[dx] == 0.f);
    }
    float4* r = reinterpret_cast<float4*>(heat + off + (size_t)dy * W);
    r[0] = make_float4(v[0], v[1], v[2], v[3]);
    r[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
  if (bad) *flag = 1;
}

extern "C" int ssp_flatten_detection_masked(const float* semi, const float* mask, int N, int Hc, int Wc, float* heat, int* flag,
                                            void* stream) {
  SSP_REQUIRE(semi && mask && heat && flag, "ssp_flatten_detection_masked: null pointer");
  SSP_REQUIRE(N > 0 && Hc > 0 && Wc > 0, "ssp_flatten_detection_masked: bad sizes N=%d Hc=%d Wc=%d", N, Hc, Wc);
  SSP_REQUIRE((((uintptr_t)heat | (uintptr_t)mask) & 15) == 0, "ssp_flatten_detection_masked: mask and output must be 16-byte aligned");
  int cells = N * Hc * Wc;
  flatten_detection_masked_kernel<<<ssp_ceil_div(cells, 128), 128, 0, (cudaStream_t)stream>>>(semi, mask, N, Hc, Wc, heat, flag);
  SSP_CUDA_CHECK_LAUNCH("flatten_detection_masked_kernel");
  return SSP_OK;
}

extern "C" int ssp_flatten_detection(const float* semi, int N, int Hc, int Wc, float* heat, void* stream) {
  SSP_REQUIRE(semi && heat, "ssp_flatten_detection: null pointer");
  SSP_REQUIRE(N > 0 && Hc > 0 && Wc > 0, "ssp_flatten_detection: bad sizes N=%d Hc=%d Wc=%d", N, Hc, Wc);
  SSP_REQUIRE(((uintptr_t)heat & 15) == 0, "ssp_flatten_detection: output must be 16-byte aligned");
  int cells = N * Hc * Wc;
  flatten_detection_kernel<<<ssp_ceil_div(cells, 128), 128, 0, (cudaStream_t)stream>>>(semi, N, Hc, Wc, heat);
  SSP_CUDA_CHECK_LAUNCH("flatten_detection_kernel");
  return SSP_OK;
}
