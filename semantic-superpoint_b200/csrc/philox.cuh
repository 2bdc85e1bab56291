// Counter-based random numbers shared by the device samplers (sparse.cu, homography.cu).  Every sampler keys Philox4x32-10
// with its seed and puts (item, purpose tag, launch counter) in the counter; the purpose tags of different samplers are kept
// disjoint, so two samplers built from the same seed draw unrelated numbers.
// Counter layout (x, y, z, w):
//   sparse.cu      (item, image << 2 | tag 0..2, launch counter lo, launch counter hi)
//   homography.cu  (homography, block << 2 | 3, launch counter lo, launch counter hi)
//   eval.cu        (problem, hypothesis, draw block, 0x80000000): the RANSAC sampler keeps no launch counter; bit 31 of the
//                  fourth word is set, which a sampler's launch counter (its high word) never reaches
#pragma once
#include <cuda_runtime.h>

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// uniform integer in [0, n) from 64 random bits (bias below n / 2^64)
__device__ __forceinline__ int uniform_below(unsigned lo, unsigned hi, int n) {
  return (int)__umul64hi(((unsigned long long)hi << 32) | lo, (unsigned long long)n);
}
