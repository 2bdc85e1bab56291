// Homography sampler on the device (SURVEY 8f rank 4): the distribution of sample_homography_np (utils/homographies.py:12-141)
// at the arguments of every call site -- shape [2, 2], shift -1, allow_artifacts True, translation_overflow 0 -- followed by
// the callers' inversion (datasets/Coco.py:345 and :271-277).  One thread per homography, float64 throughout:
//   pts1         the unit square; pts2 the centred patch of side patch_ratio, corners (0,0), (0,p), (p,p), (p,0) + margin
//   perspective  pd ~ tn(0, ay/2), hl ~ tn(0, ax/2), hr ~ tn(0, ax/2); pts2 += [[hl,pd], [hl,-pd], [hr,pd], [hr,-pd]]
//   scaling      the reference draws n_scales truncated normals, puts 1 in front of them and picks one of the first n_scales
//                uniformly: scale 1 with probability 1 / n_scales, else one tn(1, sa/2) draw -- the same law from one draw;
//                applied about the corners' mean
//   translation  per axis uniform between -min(pts2) and min(1 - pts2) (numpy's low + (high - low) u, also when low > high)
//   rotation     one of linspace(-max_angle, max_angle, n_angles) uniformly (the reference's appended 0 is never picked),
//                about the corners' mean: pts2 = (pts2 - c) [[cos, -sin], [sin, cos]] + c
//   H            getPerspectiveTransform(fp32(2 pts1 - 1), fp32(2 pts2 - 1)): the 8x8 system, partial pivoting
//   outputs      homographies = fp32(H^-1) (Coco.py:345), inv_homographies = fp32(inverse of that fp32 matrix)
//                (Coco.py:276-277); every index that is a multiple of `group` (group > 0) gets the identity (Coco.py:271)
// tn(loc, sd) = truncnorm(-2, 2, loc, sd) by its inverse CDF, loc + sd Phi^-1(Phi(-2) + u (Phi(2) - Phi(-2))) with u uniform
// in [0, 1) at 53 bits: a fixed number of draws per homography and the exact law.
// Random numbers: Philox4x32-10, key = seed, counter = (homography index, j << 2 | 3, launch counter) for the j-th four words of
// a homography (purpose tag 3; sparse.cu uses 0..2, so the two samplers draw unrelated numbers from one seed).  The seed and the
// counter come from the caller's state buffer and the last block advances the counter, as in sparse_sample_kernel.
#include "common.cuh"
#include "perspective.cuh"
#include "philox.cuh"
#include <cmath>

enum { HOMOG_PERSPECTIVE = 1, HOMOG_SCALING = 2, HOMOG_ROTATION = 4, HOMOG_TRANSLATION = 8 };
constexpr int HOMOG_THREADS = 128;

struct HomogParams {
  int flags, n_scales, n_angles, group;
  double sa, ax, ay, patch, max_angle;
};

// one homography's sequence of 64-bit draws
struct HomogDraws {
  uint2 key;
  unsigned item, clo, chi, block;
  uint4 buf;
  int left;

  __device__ unsigned long long next() {
    if (left == 0) {
      buf = philox4x32_10(make_uint4(item, (block++ << 2) | 3u, clo, chi), key);
      left = 2;
    }
    const unsigned lo = left == 2 ? buf.x : buf.z, hi = left == 2 ? buf.y : buf.w;
    --left;
    return ((unsigned long long)hi << 32) | lo;
  }
  __device__ double uniform() { return (double)(next() >> 11) * 0x1.0p-53; }
  __device__ int below(int n) {
    const unsigned long long r = next();
    return uniform_below((unsigned)r, (unsigned)(r >> 32), n);
  }
  __device__ double truncnorm2(double loc, double sd) {
    const double lo = normcdf(-2.0), hi = normcdf(2.0);
    return loc + sd * normcdfinv(lo + uniform() * (hi - lo));
  }
};

__device__ __forceinline__ void inverse3(const double (&m)[9], double (&o)[9]) {
  const double c0 = m[4] * m[8] - m[5] * m[7], c1 = m[5] * m[6] - m[3] * m[8], c2 = m[3] * m[7] - m[4] * m[6];
  const double r = 1.0 / (m[0] * c0 + m[1] * c1 + m[2] * c2);
  o[0] = c0 * r;
  o[1] = (m[2] * m[7] - m[1] * m[8]) * r;
  o[2] = (m[1] * m[5] - m[2] * m[4]) * r;
  o[3] = c1 * r;
  o[4] = (m[0] * m[8] - m[2] * m[6]) * r;
  o[5] = (m[2] * m[3] - m[0] * m[5]) * r;
  o[6] = c2 * r;
  o[7] = (m[1] * m[6] - m[0] * m[7]) * r;
  o[8] = (m[0] * m[4] - m[1] * m[3]) * r;
}

__global__ void __launch_bounds__(HOMOG_THREADS)
sample_homography_kernel(int B, HomogParams P, unsigned long long* state, float* __restrict__ hom, float* __restrict__ inv) {
  __shared__ unsigned long long s_seed, s_ctr;
  if (threadIdx.x == 0) {
    s_seed = *(volatile unsigned long long*)&state[0];
    s_ctr = *(volatile unsigned long long*)&state[1];
    // the last block to have read the launch counter advances it
    __threadfence();
    const unsigned prev = atomicInc((unsigned*)&state[2], gridDim.x - 1);  // wraps back to 0 for the next launch
    if (prev == gridDim.x - 1) state[1] = s_ctr + 1;
  }
  __syncthreads();
  const int i = blockIdx.x * HOMOG_THREADS + threadIdx.x;
  if (i >= B) return;
  double Hi[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
  if (P.group == 0 || i % P.group != 0) {
    HomogDraws d{make_uint2((unsigned)s_seed, (unsigned)(s_seed >> 32)), (unsigned)i, (unsigned)s_ctr,
                 (unsigned)(s_ctr >> 32), 0u, make_uint4(0u, 0u, 0u, 0u), 0};
    const double m = (1.0 - P.patch) / 2, e = m + P.patch;
    double px[4] = {m, m, e, e}, py[4] = {m, e, e, m};
    if (P.flags & HOMOG_PERSPECTIVE) {
      const double pd = d.truncnorm2(0.0, P.ay / 2), hl = d.truncnorm2(0.0, P.ax / 2), hr = d.truncnorm2(0.0, P.ax / 2);
      px[0] += hl; px[1] += hl; px[2] += hr; px[3] += hr;
      py[0] += pd; py[1] -= pd; py[2] += pd; py[3] -= pd;
    }
    if (P.flags & HOMOG_SCALING) {
      const int pick = d.below(P.n_scales);
      const double drawn = d.truncnorm2(1.0, P.sa / 2);
      const double s = pick == 0 ? 1.0 : drawn;
      const double cx = (((px[0] + px[1]) + px[2]) + px[3]) / 4, cy = (((py[0] + py[1]) + py[2]) + py[3]) / 4;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        px[k] = (px[k] - cx) * s + cx;
        py[k] = (py[k] - cy) * s + cy;
      }
    }
    if (P.flags & HOMOG_TRANSLATION) {
      const double tminx = fmin(fmin(px[0], px[1]), fmin(px[2], px[3]));
      const double tminy = fmin(fmin(py[0], py[1]), fmin(py[2], py[3]));
      const double tmaxx = fmin(fmin(1.0 - px[0], 1.0 - px[1]), fmin(1.0 - px[2], 1.0 - px[3]));
      const double tmaxy = fmin(fmin(1.0 - py[0], 1.0 - py[1]), fmin(1.0 - py[2], 1.0 - py[3]));
      const double tx = -tminx + (tmaxx + tminx) * d.uniform();
      const double ty = -tminy + (tmaxy + tminy) * d.uniform();
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        px[k] += tx;
        py[k] += ty;
      }
    }
    if (P.flags & HOMOG_ROTATION) {
      // numpy.linspace: start + k * (stop - start) / (n - 1), the last one exactly stop; n = 1 -> start
      const int k = d.below(P.n_angles);
      const double a = (P.n_angles > 1 && k == P.n_angles - 1)
                           ? P.max_angle
                           : __dadd_rn(__dmul_rn((double)k, (2.0 * P.max_angle) / (double)(P.n_angles > 1 ? P.n_angles - 1 : 1)),
                                       -P.max_angle);
      double sn, cs;
      sincos(a, &sn, &cs);
      const double cx = (((px[0] + px[1]) + px[2]) + px[3]) / 4, cy = (((py[0] + py[1]) + py[2]) + py[3]) / 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double dx = px[j] - cx, dy = py[j] - cy;
        px[j] = (dx * cs + dy * sn) + cx;
        py[j] = (dx * -sn + dy * cs) + cy;
      }
    }
    const float x1[4] = {-1.f, -1.f, 1.f, 1.f}, y1[4] = {-1.f, 1.f, 1.f, -1.f};
    float x2[4], y2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      x2[j] = (float)(px[j] * 2.0 - 1.0);
      y2[j] = (float)(py[j] * 2.0 - 1.0);
    }
    double H[9];
    perspective_transform(x1, y1, x2, y2, H);
    inverse3(H, Hi);
  }
  double Hf[9], Hinv[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) {
    hom[(size_t)i * 9 + c] = (float)Hi[c];
    Hf[c] = (double)(float)Hi[c];
  }
  inverse3(Hf, Hinv);
#pragma unroll
  for (int c = 0; c < 9; ++c) inv[(size_t)i * 9 + c] = (float)Hinv[c];
}

extern "C" int ssp_sample_homography(int B, int flags, int n_scales, int n_angles, double scaling_amplitude,
                                     double perspective_amplitude_x, double perspective_amplitude_y, double patch_ratio,
                                     double max_angle, int group, unsigned long long* state, float* homographies,
                                     float* inv_homographies, void* stream) {
  SSP_REQUIRE(state && homographies && inv_homographies, "ssp_sample_homography: null pointer");
  SSP_REQUIRE(B > 0 && B <= (1 << 30) && group >= 0, "ssp_sample_homography: bad sizes (B = %d, group = %d)", B, group);
  SSP_REQUIRE((flags & ~15) == 0, "ssp_sample_homography: unknown flag bits 0x%x", flags);
  SSP_REQUIRE(!(flags & HOMOG_SCALING) || n_scales > 0, "ssp_sample_homography: need n_scales > 0 (got %d)", n_scales);
  SSP_REQUIRE(!(flags & HOMOG_ROTATION) || n_angles > 0, "ssp_sample_homography: need n_angles > 0 (got %d)", n_angles);
  SSP_REQUIRE(patch_ratio > 0.0 && patch_ratio <= 1.0, "ssp_sample_homography: need 0 < patch_ratio <= 1 (got %g)",
              patch_ratio);
  SSP_REQUIRE(!(flags & HOMOG_SCALING) || (scaling_amplitude > 0.0 && std::isfinite(scaling_amplitude)),
              "ssp_sample_homography: the scaling amplitude must be positive and finite (got %g)", scaling_amplitude);
  SSP_REQUIRE(!(flags & HOMOG_PERSPECTIVE) || (perspective_amplitude_x > 0.0 && std::isfinite(perspective_amplitude_x) &&
                                               perspective_amplitude_y > 0.0 && std::isfinite(perspective_amplitude_y)),
              "ssp_sample_homography: the perspective amplitudes must be positive and finite (got %g, %g)",
              perspective_amplitude_x, perspective_amplitude_y);
  SSP_REQUIRE(!(flags & HOMOG_ROTATION) || std::isfinite(max_angle), "ssp_sample_homography: max_angle must be finite");
  const HomogParams P{flags, n_scales, n_angles, group, scaling_amplitude, perspective_amplitude_x, perspective_amplitude_y,
                      patch_ratio, max_angle};
  sample_homography_kernel<<<ssp_ceil_div(B, HOMOG_THREADS), HOMOG_THREADS, 0, (cudaStream_t)stream>>>(
      B, P, state, homographies, inv_homographies);
  SSP_CUDA_CHECK_LAUNCH("sample_homography_kernel");
  return SSP_OK;
}
