// cv2.getPerspectiveTransform in float64, shared by the homography sampler (homography.cu) and the RANSAC minimal solve
// (eval.cu): A h = b with the rows (x, y, 1, 0, 0, 0, -u x, -u y | u) and (0, 0, 0, x, y, 1, -v x, -v y | v) of the four
// correspondences (x, y) -> (u, v), partial-pivoting elimination; h33 = 1.  A zero pivot leaves a non-finite H.
// The homography sampler keeps the 8x9 matrix in registers; in ransac_score_kernel ptxas places it in a 576-byte stack
// frame (local memory), which costs little there: one solve per hypothesis against thousands of inlier tests.
#pragma once
#include <cuda_runtime.h>

template <typename T>
__device__ __forceinline__ void perspective_transform(const T (&x)[4], const T (&y)[4], const T (&u)[4], const T (&v)[4],
                                                      double (&H)[9]) {
  double a[8][9];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double X = x[i], Y = y[i], U = u[i], V = v[i];
    const double r0[9] = {X, Y, 1.0, 0.0, 0.0, 0.0, -U * X, -U * Y, U};
    const double r1[9] = {0.0, 0.0, 0.0, X, Y, 1.0, -V * X, -V * Y, V};
#pragma unroll
    for (int c = 0; c < 9; ++c) {
      a[2 * i][c] = r0[c];
      a[2 * i + 1][c] = r1[c];
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    int p = k;
    double best = fabs(a[k][k]);
#pragma unroll
    for (int r = k + 1; r < 8; ++r)
      if (fabs(a[r][k]) > best) {
        best = fabs(a[r][k]);
        p = r;
      }
#pragma unroll
    for (int r = k + 1; r < 8; ++r) {  // row swap by selects with compile-time indices, so the matrix can stay in registers
      const bool sw = r == p;
#pragma unroll
      for (int c = k; c < 9; ++c) {
        const double t = a[k][c];
        a[k][c] = sw ? a[r][c] : t;
        a[r][c] = sw ? t : a[r][c];
      }
    }
    const double piv = 1.0 / a[k][k];
#pragma unroll
    for (int r = k + 1; r < 8; ++r) {
      const double f = a[r][k] * piv;
#pragma unroll
      for (int c = k + 1; c < 9; ++c) a[r][c] -= f * a[k][c];
    }
  }
#pragma unroll
  for (int k = 7; k >= 0; --k) {
    double s = a[k][8];
#pragma unroll
    for (int c = k + 1; c < 8; ++c) s -= a[k][c] * H[c];
    H[k] = s / a[k][k];
  }
  H[8] = 1.0;
}
