// Evaluation of exported image pairs on the device: the metrics of evaluation.py (reference lineage, evaluation.py:86-499 and
// evaluations/detector_evaluation.py, evaluations/descriptor_evaluation.py) for P pairs per launch.
//
// ransac_score_kernel   grid (ceil(M / 256), n problems): the problem's matches staged in shared memory as fp32
//                       (x1, y1, x2, y2) -- exact for the integer NMS positions -- then one hypothesis per thread: 4 distinct
//                       match indices from Philox4x32-10 (key = seed, counter = (problem, hypothesis, draw block, 1 << 31)),
//                       OpenCV's sample checks (haveCollinearPoints on every triple of either image, checkSubset's orientation
//                       sign test), the 4-point solve of perspective.cuh in float64; a rejected sample scores nothing (OpenCV
//                       redraws it instead).  Each warp then counts the inliers of its 32 hypotheses over the matches,
//                       float64 arithmetic: ||pi(H p1) - p2||^2 <= thresh^2, |w| <= FLT_EPSILON an outlier.
// ransac_refit_kernel   one block per problem: the hypothesis with the most inliers (lowest index on ties), its inlier mask,
//                       and the refit on those inliers: OpenCV's normalised DLT (centroid and mean absolute deviation per
//                       axis, the eigenvector of the smallest eigenvalue of the 9x9 L^T L by cyclic Jacobi), h33 = 1.
//                       OpenCV follows that DLT with 10 Levenberg-Marquardt iterations; this estimator does not.
// eval_repeatability_kernel, eval_metrics_kernel   one block per pair (see the header for the definitions).
#include "common.cuh"
#include "perspective.cuh"
#include "philox.cuh"
#include <algorithm>
#include <cfloat>

#define SSP_RANSAC_MAX_MATCHES 8192

namespace {

constexpr int EV_THREADS = 256;
constexpr int EV_WARPS = EV_THREADS / 32;
constexpr unsigned RANSAC_TAG = 0x80000000u;  // fourth counter word: disjoint from the samplers' launch counters (philox.cuh)
constexpr double GT_INLIER_DIST = 3.0;        // getInliers' epi of evaluation.py (map_inliers "gt")

// Ordered compaction of a pair's match list [3, Lmax] (index 1, index 2, distance): the first L0 matches, or with
// `subset` those whose distance is below subset_dist.  store(k, off) is called for the k-th match kept, at position off in
// increasing k order.  Every thread of the block must call it; returns the number kept (the same in every thread).
template <class F>
__device__ int compact_matches(const double* __restrict__ m, int Lmax, int L0, bool subset, double subset_dist, int* wcount,
                               F store) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int base = 0;
  for (int k0 = 0; k0 < L0; k0 += EV_THREADS) {
    const int k = k0 + threadIdx.x;
    const bool keep = k < L0 && (!subset || m[2 * (size_t)Lmax + k] < subset_dist);
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wcount[warp] = __popc(bal);
    __syncthreads();
    int off = base, tot = 0;
    for (int w = 0; w < EV_WARPS; ++w) {
      if (w < warp) off += wcount[w];
      tot += wcount[w];
    }
    if (keep) store(k, off + __popc(bal & ((1u << lane) - 1u)));
    base += tot;
    __syncthreads();
  }
  return base;
}

struct RansacArgs {
  const double* pts1;  // [P, 3, cap1] (x, y, conf) rows
  const double* pts2;  // [P, 3, cap2]
  int cap1, cap2;
  const double* matches;       // [P, 3, Lmax]
  const unsigned int* nmatch;  // [P]
  int Lmax, P, M;
  double subset_dist, t2;
  unsigned long long seed;
  int* count;       // [n, M] inliers per hypothesis, -1 = rejected sample
  double* hyp;      // [n, M, 9] hypotheses (NaN when rejected)
  int* samples;     // [n, M, 4] or NULL
  double* H;        // [n, 9]
  int* ninl;        // [n]
  uint8_t* mask;    // [n, Lmax]
  int* best;        // [n]
};

// problem q = set * P + p: the matches of pair p, all of them (set 0) or those closer than subset_dist (set 1), staged
__device__ int stage_problem(const RansacArgs& a, int q, float4* s, int* wcount) {
  const int p = q % a.P;
  const double* m = a.matches + (size_t)p * 3 * a.Lmax;
  const double* p1 = a.pts1 + (size_t)p * 3 * a.cap1;
  const double* p2 = a.pts2 + (size_t)p * 3 * a.cap2;
  const int L0 = min((int)__ldg(a.nmatch + p), a.Lmax);
  return compact_matches(m, a.Lmax, L0, q >= a.P, a.subset_dist, wcount, [&](int k, int off) {
    const int i = (int)m[k], j = (int)m[(size_t)a.Lmax + k];
    s[off] = make_float4((float)p1[i], (float)p1[(size_t)a.cap1 + i], (float)p2[j], (float)p2[(size_t)a.cap2 + j]);
  });
}

__device__ __forceinline__ bool is_inlier(const double (&h)[9], float4 m, double t2) {
  const double x = m.x, y = m.y;
  const double w = fma(h[7], y, fma(h[6], x, h[8]));
  if (!(fabs(w) > (double)FLT_EPSILON)) return false;
  const double iw = 1.0 / w;
  const double dx = fma(fma(h[1], y, fma(h[0], x, h[2])), iw, -(double)m.z);
  const double dy = fma(fma(h[4], y, fma(h[3], x, h[5])), iw, -(double)m.w);
  return fma(dx, dx, dy * dy) <= t2;
}

// 4 distinct indices in [0, L): the k-th draw picks uniformly among the L - k indices not taken yet
__device__ __forceinline__ void draw4(unsigned long long seed, int q, int h, int L, int (&idx)[4]) {
  const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  const uint4 r0 = philox4x32_10(make_uint4((unsigned)q, (unsigned)h, 0u, RANSAC_TAG), key);
  const uint4 r1 = philox4x32_10(make_uint4((unsigned)q, (unsigned)h, 1u, RANSAC_TAG), key);
  const unsigned lo[4] = {r0.x, r0.z, r1.x, r1.z}, hi[4] = {r0.y, r0.w, r1.y, r1.w};
  int srt[4];  // taken so far, ascending
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int v = uniform_below(lo[k], hi[k], L - k);
#pragma unroll
    for (int t = 0; t < k; ++t) v += srt[t] <= v;
    idx[k] = v;
    int pos = k;
#pragma unroll
    for (int t = k - 1; t >= 0; --t)
      if (srt[t] > v) { srt[t + 1] = srt[t]; pos = t; }
    srt[pos] = v;
  }
}

// OpenCV haveCollinearPoints, over every triple of the four points (float differences, as on Point2f)
__device__ __forceinline__ bool collinear(const float (&x)[4], const float (&y)[4]) {
  bool c = false;
#pragma unroll
  for (int i = 2; i < 4; ++i)
#pragma unroll
    for (int j = 1; j < i; ++j)
#pragma unroll
      for (int k = 0; k < j; ++k) {
        const double dx1 = x[j] - x[i], dy1 = y[j] - y[i], dx2 = x[k] - x[i], dy2 = y[k] - y[i];
        const double cr = __dsub_rn(__dmul_rn(dx2, dy1), __dmul_rn(dy2, dx1));
        c |= fabs(cr) <= (double)FLT_EPSILON * (((fabs(dx1) + fabs(dy1)) + fabs(dx2)) + fabs(dy2));
      }
  return c;
}

// determinant of [[xa, ya, 1], [xb, yb, 1], [xc, yc, 1]] in cv::determinant(Matx33d)'s order
__device__ __forceinline__ double det3(double xa, double ya, double xb, double yb, double xc, double yc) {
  const double t0 = __dmul_rn(xa, __dsub_rn(yb, yc));
  const double t1 = __dmul_rn(ya, __dsub_rn(xb, xc));
  const double t2 = __dsub_rn(__dmul_rn(xb, yc), __dmul_rn(xc, yb));
  return __dadd_rn(__dsub_rn(t0, t1), t2);
}

// checkSubset's orientation test: the four triangle-orientation products all positive or all negative
__device__ __forceinline__ bool orientation_ok(const float (&x1)[4], const float (&y1)[4], const float (&x2)[4],
                                               const float (&y2)[4]) {
  const int tt[4][3] = {{0, 1, 2}, {1, 2, 3}, {0, 2, 3}, {0, 1, 3}};
  int neg = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = tt[i][0], b = tt[i][1], c = tt[i][2];
    const double dA = det3(x1[a], y1[a], x1[b], y1[b], x1[c], y1[c]);
    const double dB = det3(x2[a], y2[a], x2[b], y2[b], x2[c], y2[c]);
    neg += __dmul_rn(dA, dB) < 0.0;
  }
  return neg == 0 || neg == 4;
}

__global__ void __launch_bounds__(EV_THREADS) ransac_score_kernel(const RansacArgs a) {
  extern __shared__ float4 s_m[];  // [Lmax]
  __shared__ double s_h[EV_THREADS][9];
  __shared__ bool s_ok[EV_THREADS];
  __shared__ int wcount[EV_WARPS];
  const int q = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = stage_problem(a, q, s_m, wcount);
  const int h = blockIdx.x * EV_THREADS + threadIdx.x;
  bool ok = false;
  if (h < a.M) {
    int idx[4] = {-1, -1, -1, -1};
    double H[9];
    if (L >= 4) {
      draw4(a.seed, q, h, L, idx);
      float x1[4], y1[4], x2[4], y2[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 m = s_m[idx[k]];
        x1[k] = m.x; y1[k] = m.y; x2[k] = m.z; y2[k] = m.w;
      }
      if (!collinear(x1, y1) && !collinear(x2, y2) && orientation_ok(x1, y1, x2, y2)) {
        perspective_transform(x1, y1, x2, y2, H);
        ok = true;
#pragma unroll
        for (int c = 0; c < 9; ++c) ok &= isfinite(H[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 9; ++c) s_h[threadIdx.x][c] = ok ? H[c] : __longlong_as_double(0x7ff8000000000000ll);
    if (a.samples) {
      int* o = a.samples + ((size_t)q * a.M + h) * 4;
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k] = idx[k];
    }
  }
  s_ok[threadIdx.x] = ok;
  __syncwarp();
  // the warp counts the inliers of its 32 hypotheses, one after the other, the lanes striding over the matches
  for (int k = 0; k < 32; ++k) {
    const int t = warp * 32 + k, hh = blockIdx.x * EV_THREADS + t;
    if (hh >= a.M) break;
    const size_t o = (size_t)q * a.M + hh;
    int cnt = -1;
    if (s_ok[t]) {
      double Hk[9];
#pragma unroll
      for (int c = 0; c < 9; ++c) Hk[c] = s_h[t][c];
      int c = 0;
      for (int j = lane; j < L; j += 32) c += is_inlier(Hk, s_m[j], a.t2);
      cnt = __reduce_add_sync(0xffffffffu, c);
    }
    if (lane == 0) a.count[o] = cnt;
    if (lane < 9) a.hyp[o * 9 + lane] = s_h[t][lane];
  }
}

// cyclic Jacobi on the symmetric 9x9 matrix A (shared memory), run by one warp; V receives the eigenvectors as columns
__device__ void jacobi9(double (*A)[9], double (*V)[9]) {
  const int lane = threadIdx.x & 31;
  if (lane < 9)
    for (int c = 0; c < 9; ++c) V[lane][c] = lane == c ? 1.0 : 0.0;
  __syncwarp();
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, fro = 0.0;
    for (int p = 0; p < 9; ++p)
      for (int q = 0; q < 9; ++q) {
        const double v = A[p][q] * A[p][q];
        fro += v;
        if (p != q) off += v;
      }
    if (!(off > 1e-36 * fro)) break;
    for (int p = 0; p < 8; ++p)
      for (int q = p + 1; q < 9; ++q) {
        const double apq = A[p][q];
        if (apq == 0.0) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        __syncwarp();
        if (lane < 9) {
          const double akp = A[lane][p], akq = A[lane][q];
          A[lane][p] = c * akp - s * akq;
          A[lane][q] = s * akp + c * akq;
        }
        __syncwarp();
        if (lane < 9) {
          const double apk = A[p][lane], aqk = A[q][lane];
          A[p][lane] = c * apk - s * aqk;
          A[q][lane] = s * apk + c * aqk;
          const double vkp = V[lane][p], vkq = V[lane][q];
          V[lane][p] = c * vkp - s * vkq;
          V[lane][q] = s * vkp + c * vkq;
        }
        __syncwarp();
      }
  }
}

__global__ void __launch_bounds__(EV_THREADS) ransac_refit_kernel(const RansacArgs a) {
  extern __shared__ float4 s_m[];                  // [Lmax]
  uint8_t* s_in = reinterpret_cast<uint8_t*>(s_m + a.Lmax);  // [Lmax] inlier flags
  __shared__ double red[32];
  __shared__ double s_part[EV_WARPS][45];
  __shared__ double s_A[9][9], s_V[9][9];
  __shared__ double s_stat[8];
  __shared__ unsigned long long s_key[EV_WARPS];
  __shared__ bool s_fit;
  __shared__ double s_Hout[9];
  __shared__ int wcount[EV_WARPS];
  const int q = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  const int L = stage_problem(a, q, s_m, wcount);
  // best hypothesis: most inliers, then lowest index
  unsigned long long key = 0;
  for (int h = tid; h < a.M; h += EV_THREADS) {
    const int c = a.count[(size_t)q * a.M + h];
    const unsigned long long k = ((unsigned long long)(unsigned)(c + 1) << 32) | (unsigned)(a.M - 1 - h);
    key = k > key ? k : key;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, key, o);
    key = v > key ? v : key;
  }
  if (lane == 0) s_key[warp] = key;
  __syncthreads();
  key = 0;
  for (int w = 0; w < EV_WARPS; ++w) key = s_key[w] > key ? s_key[w] : key;
  const int best_cnt = (int)(key >> 32) - 1, best_h = a.M - 1 - (int)(key & 0xffffffffu);
  const bool have = L >= 4 && best_cnt >= 4;
  double H[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) H[c] = have ? a.hyp[((size_t)q * a.M + best_h) * 9 + c] : 0.0;
  // inlier flags and the sums of the normalisation
  double sx1 = 0.0, sy1 = 0.0, sx2 = 0.0, sy2 = 0.0, n = 0.0;
  for (int k = tid; k < a.Lmax; k += EV_THREADS) {
    const bool in = have && k < L && is_inlier(H, s_m[k], a.t2);
    s_in[k] = in;
    if (in) {
      const float4 m = s_m[k];
      sx1 += m.x; sy1 += m.y; sx2 += m.z; sy2 += m.w; n += 1.0;
    }
  }
  const double tot[5] = {sx1, sy1, sx2, sy2, n};
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const double r = block_sum_d(tot[i], red);
    if (tid == 0) s_stat[i] = r;
  }
  __syncthreads();
  const double cnt = s_stat[4];
  const double c1x = s_stat[0] / cnt, c1y = s_stat[1] / cnt, c2x = s_stat[2] / cnt, c2y = s_stat[3] / cnt;
  double ax1 = 0.0, ay1 = 0.0, ax2 = 0.0, ay2 = 0.0;
  for (int k = tid; k < L; k += EV_THREADS)
    if (s_in[k]) {
      const float4 m = s_m[k];
      ax1 += fabs(m.x - c1x); ay1 += fabs(m.y - c1y); ax2 += fabs(m.z - c2x); ay2 += fabs(m.w - c2y);
    }
  const double dev[4] = {ax1, ay1, ax2, ay2};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double r = block_sum_d(dev[i], red);
    if (tid == 0) s_stat[i] = r;
  }
  __syncthreads();
  const bool fit = have && s_stat[0] >= DBL_EPSILON && s_stat[1] >= DBL_EPSILON && s_stat[2] >= DBL_EPSILON &&
                   s_stat[3] >= DBL_EPSILON;
  // L^T L of the normalised correspondences (upper triangle, 45 entries): per-thread partial sums, then the block's
  const double s1x = cnt / s_stat[0], s1y = cnt / s_stat[1], s2x = cnt / s_stat[2], s2y = cnt / s_stat[3];
  double acc[45];
#pragma unroll
  for (int i = 0; i < 45; ++i) acc[i] = 0.0;
  if (fit)
    for (int k = tid; k < L; k += EV_THREADS)
      if (s_in[k]) {
        const float4 m = s_m[k];
        const double X = (m.x - c1x) * s1x, Y = (m.y - c1y) * s1y, x = (m.z - c2x) * s2x, y = (m.w - c2y) * s2y;
        const double Lx[9] = {X, Y, 1.0, 0.0, 0.0, 0.0, -x * X, -x * Y, -x};
        const double Ly[9] = {0.0, 0.0, 0.0, X, Y, 1.0, -y * X, -y * Y, -y};
        int e = 0;
#pragma unroll
        for (int r = 0; r < 9; ++r)
#pragma unroll
          for (int c = r; c < 9; ++c) acc[e++] += Lx[r] * Lx[c] + Ly[r] * Ly[c];
      }
#pragma unroll
  for (int i = 0; i < 45; ++i) {
    const double v = warp_sum_d(acc[i]);
    if (lane == 0) s_part[warp][i] = v;
  }
  __syncthreads();
  if (tid < 45) {
    double v = 0.0;
    for (int w = 0; w < EV_WARPS; ++w) v += s_part[w][tid];
    int r = 0, e = tid;
    while (e >= 9 - r) { e -= 9 - r; ++r; }
    s_A[r][r + e] = v;
    s_A[r + e][r] = v;
  }
  __syncthreads();
  if (warp == 0) {
    if (fit) jacobi9(s_A, s_V);
    if (lane == 0) {
      int imin = 0;
      for (int i = 1; i < 9; ++i)
        if (s_A[i][i] < s_A[imin][imin]) imin = i;
      double h0[9];
      for (int i = 0; i < 9; ++i) h0[i] = s_V[i][imin];
      // H = invHnorm(image 2) * H0 * Hnorm(image 1), then h33 = 1
      const double inv2[9] = {1.0 / s2x, 0.0, c2x, 0.0, 1.0 / s2y, c2y, 0.0, 0.0, 1.0};
      const double n1[9] = {s1x, 0.0, -c1x * s1x, 0.0, s1y, -c1y * s1y, 0.0, 0.0, 1.0};
      double t[9], r[9];
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
          t[i * 3 + j] = inv2[i * 3] * h0[j] + inv2[i * 3 + 1] * h0[3 + j] + inv2[i * 3 + 2] * h0[6 + j];
        }
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) r[i * 3 + j] = t[i * 3] * n1[j] + t[i * 3 + 1] * n1[3 + j] + t[i * 3 + 2] * n1[6 + j];
      bool ok = fit;
      for (int i = 0; i < 9; ++i) {
        s_Hout[i] = r[i] / r[8];
        ok &= isfinite(s_Hout[i]);
      }
      s_fit = ok;
    }
  }
  __syncthreads();
  const bool est = s_fit;
  if (tid < 9) a.H[(size_t)q * 9 + tid] = est ? s_Hout[tid] : __longlong_as_double(0x7ff8000000000000ll);
  if (tid == 0) {
    a.ninl[q] = est ? (int)cnt : 0;
    a.best[q] = est ? best_h : -1;
  }
  for (int k = tid; k < a.Lmax; k += EV_THREADS) a.mask[(size_t)q * a.Lmax + k] = est ? s_in[k] : 0;
}

struct PairArgs {
  const double* pts1;  // [P, 3, cap1]
  const double* pts2;  // [P, 3, cap2]
  int cap1, cap2;
  const unsigned int* counts1;  // [P]; pair p uses its first min(counts[p], limit) points
  const unsigned int* counts2;
  int limit, P;
  const double* Hs;  // [P, 2, 9]: H (image 1 -> image 2, pixels) and H^-1
  double Himg, Wimg;
};

__device__ __forceinline__ int eff(const unsigned int* c, int p, int limit) {
  const unsigned v = __ldg(c + p);
  return v < (unsigned)limit ? (int)v : limit;
}

// squared distance with numpy's rounding (no contraction): dx * dx + dy * dy
__device__ __forceinline__ double dist2(double ax, double ay, double bx, double by) {
  const double dx = __dsub_rn(ax, bx), dy = __dsub_rn(ay, by);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}

__device__ __forceinline__ bool in_image(double x, double y, double W, double H) {
  return x >= 0.0 && x < W && y >= 0.0 && y < H;
}

__global__ void __launch_bounds__(EV_THREADS)
eval_repeatability_kernel(const PairArgs a, int keep_k, double thresh, double* __restrict__ out) {
  extern __shared__ double2 s_sel[];  // [ksel1 + ksel2], then the keep flags [cap1 + cap2]
  __shared__ double red[32];
  __shared__ int s_n[2];
  const int p = blockIdx.x, tid = threadIdx.x;
  const int ksel1 = min(keep_k, a.cap1), ksel2 = min(keep_k, a.cap2);
  double2* sel[2] = {s_sel, s_sel + ksel1};
  uint8_t* keep[2] = {reinterpret_cast<uint8_t*>(s_sel + ksel1 + ksel2), reinterpret_cast<uint8_t*>(s_sel + ksel1 + ksel2) + a.cap1};
  const double* pts[2] = {a.pts1 + (size_t)p * 3 * a.cap1, a.pts2 + (size_t)p * 3 * a.cap2};
  const int cap[2] = {a.cap1, a.cap2};
  const int n[2] = {eff(a.counts1, p, a.limit), eff(a.counts2, p, a.limit)};
  const double* H = a.Hs + (size_t)p * 18;
  // side 0: the true warps of image 1's points by H, kept inside image 2; side 1: image 2's points whose back-warp by
  // H^-1 lies inside image 1, at their own coordinates (keep_true_keypoints)
  for (int s = 0; s < 2; ++s)
    for (int i = tid; i < n[s]; i += EV_THREADS) {
      double ox, oy;
      warp_keypoint_f64(s == 0 ? H : H + 9, pts[s][i], pts[s][cap[s] + i], ox, oy);
      keep[s][i] = in_image(ox, oy, a.Wimg, a.Himg);
    }
  __syncthreads();
  // select_k_best: the keep_k most confident kept points, ties at the cut resolved as a stable argsort would (the later
  // index counts as more confident); each selected point goes to the slot of its rank
  int nsel[2];
  for (int s = 0; s < 2; ++s) {
    int kept = 0;
    for (int i = tid; i < n[s]; i += EV_THREADS) {
      if (!keep[s][i]) continue;
      ++kept;
      const double ci = pts[s][2 * (size_t)cap[s] + i];
      int rank = 0;
      for (int j = 0; j < n[s] && rank < keep_k; ++j) {
        if (!keep[s][j]) continue;
        const double cj = __ldg(pts[s] + 2 * (size_t)cap[s] + j);
        rank += cj > ci || (cj == ci && j > i);
      }
      if (rank < keep_k) {
        double x = pts[s][i], y = pts[s][cap[s] + i];
        if (s == 0) warp_keypoint_f64(H, pts[s][i], pts[s][cap[s] + i], x, y);
        sel[s][rank] = make_double2(x, y);
      }
    }
    const double k = block_sum_d((double)kept, red);
    if (tid == 0) s_n[s] = min((int)k, keep_k);
    __syncthreads();
    nsel[s] = s_n[s];
  }
  // mutual nearest distances <= thresh, both ways
  double cnt[2] = {0.0, 0.0}, err[2] = {0.0, 0.0};
  for (int s = 0; s < 2; ++s) {
    if (nsel[1 - s] == 0) continue;
    for (int i = tid; i < nsel[s]; i += EV_THREADS) {
      const double2 u = sel[s][i];
      double best = INFINITY;
      for (int j = 0; j < nsel[1 - s]; ++j) {
        const double2 v = sel[1 - s][j];
        best = fmin(best, dist2(u.x, u.y, v.x, v.y));
      }
      const double d = sqrt(best);
      if (d <= thresh) { cnt[s] += 1.0; err[s] += d; }
    }
  }
  const double c0 = block_sum_d(cnt[0], red), c1 = block_sum_d(cnt[1], red);
  const double e0 = block_sum_d(err[0], red), e1 = block_sum_d(err[1], red);
  if (tid == 0) {
    const double c = c0 + c1;
    const int N = nsel[0] + nsel[1];
    out[2 * (size_t)p] = (c > 0.0 && N > 0) ? c / N : 0.0;
    out[2 * (size_t)p + 1] = c > 0.0 ? e0 / c + e1 / c : -1.0;
  }
}

struct MetricArgs {
  const double* matches;       // [P, 3, Lmax] the cross-check matches
  const unsigned int* nmatch;  // [P]
  int Lmax;
  double subset_dist;    // the mAP matches: distance below this
  const double* H_est;   // [n, 9], NaN = no estimate
  const int* ninl;       // [n]
  const uint8_t* mask;   // [n, Lmax]; problems P.. are the mAP matches' RANSAC (map_gt == 0)
  int map_gt, T;
  double thr[8];
};

__global__ void __launch_bounds__(EV_THREADS)
eval_metrics_kernel(const PairArgs a, const MetricArgs b, double* __restrict__ out) {
  extern __shared__ double s_d[];  // [Lmax] distances of the mAP matches, then their labels [Lmax]
  uint8_t* s_lab = reinterpret_cast<uint8_t*>(s_d + b.Lmax);
  __shared__ double red[32];
  __shared__ int wcount[EV_WARPS];
  const int p = blockIdx.x, tid = threadIdx.x;
  const double* p1 = a.pts1 + (size_t)p * 3 * a.cap1;
  const double* p2 = a.pts2 + (size_t)p * 3 * a.cap2;
  const int n1 = eff(a.counts1, p, a.limit), n2 = eff(a.counts2, p, a.limit);
  const double* H = a.Hs + (size_t)p * 18;
  // K2': image 2's points whose back-warp lies in the image, with warpLabels' arithmetic (integer-truncated points, fp32
  // warp in warp_points_mask_kernel's order, filter_points' inclusive bounds)
  float hi[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) hi[c] = (float)H[9 + c];
  double k2 = 0.0;
  for (int j = tid; j < n2; j += EV_THREADS) {
    float ox, oy;
    homography_apply(hi, (float)trunc(p2[j]), (float)trunc(p2[a.cap2 + j]), ox, oy);
    k2 += (ox >= 0.f && ox <= (float)a.Wimg - 1.f && oy >= 0.f && oy <= (float)a.Himg - 1.f) ? 1.0 : 0.0;
  }
  k2 = block_sum_d(k2, red);
  // the mAP matches and their labels
  const double* m = b.matches + (size_t)p * 3 * b.Lmax;
  const int L0 = min((int)__ldg(b.nmatch + p), b.Lmax);
  const uint8_t* mk = b.mask + (size_t)(a.P + p) * b.Lmax;
  const int L = compact_matches(m, b.Lmax, L0, true, b.subset_dist, wcount, [&](int k, int off) {
    s_d[off] = m[2 * (size_t)b.Lmax + k];
    bool lab;
    if (b.map_gt) {
      const int i = (int)m[k], j = (int)m[(size_t)b.Lmax + k];
      double ox, oy;
      warp_keypoint_f64(H, p1[i], p1[a.cap1 + i], ox, oy);
      lab = sqrt(dist2(ox, oy, p2[j], p2[a.cap2 + j])) < GT_INLIER_DIST;
    } else {
      lab = mk[off];
    }
    s_lab[off] = lab;
  });
  // average precision with score = -distance: (1 / #pos) sum over positives i of TP(d <= d_i) / N(d <= d_i)
  double num = 0.0, pos = 0.0;
  for (int i = tid; i < L; i += EV_THREADS) {
    if (!s_lab[i]) continue;
    pos += 1.0;
    const double di = s_d[i];
    int tp = 0, all = 0;
    for (int j = 0; j < L; ++j) {
      const bool le = s_d[j] <= di;
      all += le;
      tp += le && s_lab[j];
    }
    num += (double)tp / (double)all;
  }
  num = block_sum_d(num, red);
  pos = block_sum_d(pos, red);
  if (tid == 0) {
    double* o = out + (size_t)p * (3 + b.T);
    const double* He = b.H_est + (size_t)p * 9;
    double md = He[8] == He[8] ? 0.0 : __longlong_as_double(0x7ff8000000000000ll);
    if (md == 0.0) {
      const double cx[4] = {0.0, 0.0, a.Wimg - 1.0, a.Wimg - 1.0}, cy[4] = {0.0, a.Himg - 1.0, 0.0, a.Himg - 1.0};
      for (int c = 0; c < 4; ++c) {
        double rx, ry, ex, ey;
        warp_keypoint_f64(H, cx[c], cy[c], rx, ry);
        warp_keypoint_f64(He, cx[c], cy[c], ex, ey);
        md = __dadd_rn(md, sqrt(dist2(rx, ry, ex, ey)));
      }
      md = md / 4.0;
    }
    o[0] = md;
    o[1] = n1 + k2 > 0.0 ? 2.0 * b.ninl[p] / (n1 + k2) : 0.0;
    o[2] = pos > 0.0 ? num / pos : 0.0;
    for (int t = 0; t < b.T; ++t) o[3 + t] = md <= b.thr[t] ? 1.0 : 0.0;
  }
}

int pair_args(PairArgs& a, const char* fn, const double* pts1, int cap1, const unsigned int* counts1, const double* pts2,
              int cap2, const unsigned int* counts2, int limit, int P, const double* Hs, int Himg, int Wimg) {
  SSP_REQUIRE(pts1 && counts1 && pts2 && counts2 && Hs, "%s: null pointer", fn);
  SSP_REQUIRE(P > 0 && P <= 65535 && cap1 > 0 && cap2 > 0 && limit > 0 && Himg > 0 && Wimg > 0,
              "%s: bad sizes P=%d cap1=%d cap2=%d limit=%d shape=(%d, %d)", fn, P, cap1, cap2, limit, Himg, Wimg);
  SSP_REQUIRE(limit <= cap1 && limit <= cap2, "%s: limit=%d exceeds a point capacity (cap1=%d, cap2=%d)", fn, limit, cap1,
              cap2);
  a.pts1 = pts1; a.pts2 = pts2; a.cap1 = cap1; a.cap2 = cap2; a.counts1 = counts1; a.counts2 = counts2;
  a.limit = limit; a.P = P; a.Hs = Hs; a.Himg = Himg; a.Wimg = Wimg;
  return SSP_OK;
}

}  // namespace

extern "C" size_t ssp_ransac_homography_ws_bytes(int n, int M) {
  return (n > 0 && M > 0) ? (size_t)n * M * (9 * sizeof(double) + sizeof(int)) : 0;
}

extern "C" int ssp_ransac_homography(const double* pts1, int cap1, const double* pts2, int cap2, const double* matches,
                                     const unsigned int* nmatch, int Lmax, int P, int n_sets, double subset_dist, int M,
                                     double thresh, unsigned long long seed, double* H, int* ninl, unsigned char* mask,
                                     int* best, int* samples, int* hyp_inliers, void* ws, size_t ws_bytes, void* stream) {
  SSP_REQUIRE(pts1 && pts2 && matches && nmatch && H && ninl && mask && best && ws, "ssp_ransac_homography: null pointer");
  SSP_REQUIRE(P > 0 && P <= 32767 && cap1 > 0 && cap2 > 0 && (n_sets == 1 || n_sets == 2),
              "ssp_ransac_homography: bad sizes P=%d cap1=%d cap2=%d n_sets=%d", P, cap1, cap2, n_sets);
  SSP_REQUIRE(Lmax > 0 && Lmax <= SSP_RANSAC_MAX_MATCHES,
              "ssp_ransac_homography: Lmax=%d matches per problem, the limit is %d", Lmax, SSP_RANSAC_MAX_MATCHES);
  SSP_REQUIRE(M > 0 && M <= (1 << 24), "ssp_ransac_homography: need 0 < M <= 2^24 hypotheses (got %d)", M);
  SSP_REQUIRE(thresh > 0.0 && thresh < INFINITY, "ssp_ransac_homography: the threshold must be positive and finite");
  const int n = n_sets * P;
  SSP_REQUIRE(ws_bytes >= ssp_ransac_homography_ws_bytes(n, M), "ssp_ransac_homography: workspace too small");
  SSP_REQUIRE(((uintptr_t)ws & 7) == 0, "ssp_ransac_homography: the workspace must be 8-byte aligned");
  RansacArgs a;
  a.pts1 = pts1; a.pts2 = pts2; a.cap1 = cap1; a.cap2 = cap2; a.matches = matches; a.nmatch = nmatch;
  a.Lmax = Lmax; a.P = P; a.M = M; a.subset_dist = subset_dist; a.t2 = thresh * thresh; a.seed = seed;
  a.hyp = reinterpret_cast<double*>(ws);
  a.count = hyp_inliers ? hyp_inliers : reinterpret_cast<int*>(a.hyp + (size_t)n * M * 9);
  a.samples = samples; a.H = H; a.ninl = ninl; a.mask = mask; a.best = best;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t sm_score = (size_t)Lmax * sizeof(float4), sm_refit = (size_t)Lmax * (sizeof(float4) + 1);
  SSP_CUDA_CALL(cudaFuncSetAttribute(ransac_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_score));
  SSP_CUDA_CALL(cudaFuncSetAttribute(ransac_refit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_refit));
  ransac_score_kernel<<<dim3(ssp_ceil_div(M, EV_THREADS), n), EV_THREADS, sm_score, st>>>(a);
  SSP_CUDA_CHECK_LAUNCH("ransac_score_kernel");
  ransac_refit_kernel<<<n, EV_THREADS, sm_refit, st>>>(a);
  SSP_CUDA_CHECK_LAUNCH("ransac_refit_kernel");
  return SSP_OK;
}

extern "C" int ssp_eval_repeatability(const double* pts1, int cap1, const unsigned int* counts1, const double* pts2,
                                      int cap2, const unsigned int* counts2, int limit, int P, const double* Hs, int Himg,
                                      int Wimg, int keep_k, double dist_thresh, double* out, void* stream) {
  PairArgs a;
  int rc = pair_args(a, "ssp_eval_repeatability", pts1, cap1, counts1, pts2, cap2, counts2, limit, P, Hs, Himg, Wimg);
  if (rc) return rc;
  SSP_REQUIRE(out, "ssp_eval_repeatability: null pointer");
  SSP_REQUIRE(keep_k > 0 && dist_thresh >= 0.0, "ssp_eval_repeatability: need keep_k > 0 and dist_thresh >= 0");
  const size_t smem = ((size_t)std::min(keep_k, cap1) + std::min(keep_k, cap2)) * sizeof(double2) + cap1 + cap2;
  SSP_REQUIRE(smem <= 200 * 1024, "ssp_eval_repeatability: min(keep_k, cap) = %d, %d points too many for shared memory",
              std::min(keep_k, cap1), std::min(keep_k, cap2));
  SSP_CUDA_CALL(cudaFuncSetAttribute(eval_repeatability_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  eval_repeatability_kernel<<<P, EV_THREADS, smem, (cudaStream_t)stream>>>(a, keep_k, dist_thresh, out);
  SSP_CUDA_CHECK_LAUNCH("eval_repeatability_kernel");
  return SSP_OK;
}

extern "C" int ssp_eval_match_metrics(const double* pts1, int cap1, const unsigned int* counts1, const double* pts2,
                                      int cap2, const unsigned int* counts2, int limit, int P, const double* Hs, int Himg,
                                      int Wimg, const double* matches, const unsigned int* nmatch, int Lmax,
                                      double subset_dist, const double* H_est, const int* ninl, const unsigned char* mask,
                                      int map_gt, const double* correctness_thresh, int T, double* out, void* stream) {
  PairArgs a;
  int rc = pair_args(a, "ssp_eval_match_metrics", pts1, cap1, counts1, pts2, cap2, counts2, limit, P, Hs, Himg, Wimg);
  if (rc) return rc;
  SSP_REQUIRE(matches && nmatch && H_est && ninl && mask && correctness_thresh && out,
              "ssp_eval_match_metrics: null pointer");
  SSP_REQUIRE(Lmax > 0 && Lmax <= SSP_RANSAC_MAX_MATCHES, "ssp_eval_match_metrics: Lmax=%d, the limit is %d", Lmax,
              SSP_RANSAC_MAX_MATCHES);
  SSP_REQUIRE(T > 0 && T <= 8, "ssp_eval_match_metrics: 1 to 8 correctness thresholds (got %d)", T);
  SSP_REQUIRE(map_gt == 0 || map_gt == 1, "ssp_eval_match_metrics: map_gt is 0 (RANSAC labels) or 1 (ground truth)");
  MetricArgs b;
  b.matches = matches; b.nmatch = nmatch; b.Lmax = Lmax; b.subset_dist = subset_dist; b.H_est = H_est; b.ninl = ninl;
  b.mask = mask; b.map_gt = map_gt; b.T = T;
  for (int t = 0; t < 8; ++t) b.thr[t] = t < T ? correctness_thresh[t] : 0.0;  // host array, read at launch
  const size_t smem = (size_t)Lmax * (sizeof(double) + 1);
  SSP_CUDA_CALL(cudaFuncSetAttribute(eval_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  eval_metrics_kernel<<<P, EV_THREADS, smem, (cudaStream_t)stream>>>(a, b, out);
  SSP_CUDA_CHECK_LAUNCH("eval_metrics_kernel");
  return SSP_OK;
}
