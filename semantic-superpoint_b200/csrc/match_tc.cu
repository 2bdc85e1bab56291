// Two-way nearest-neighbour matching of a batch of keypoint pairs on the tensor cores (sm_100a): the batched form of
// PointTracker.nn_match_two_way (models/model_wrap.py:451-494) that the descriptor export runs once per image pair.
//
// Operands are ssp_desc_pack's bf16 hi / lo planes [P, R, 256] of the two descriptor sets (the loss's bf16x3 format): three
// MMA chains hi*hi + lo*hi + hi*lo give fp32-grade dot products.  The K1 x K2 distance matrix never reaches memory.
//
// nn_match_tc_kernel, persistent, one CTA per SM, work item = (pair p, 128-row tile mt of image-1 points, 128-column tile nt
// of image-2 points) over the tiles that hold points (a pair with n1 x n2 points costs ceil(n1/128) x ceil(n2/128) items):
//   warp 8      TMA producer: the item's 128 A rows, all 256 channels of both planes, resident while the row tile stays
//               (4 boxes of [64 ch x 128 rows x 2 planes]); B ring of NS such boxes
//   warp 9      MMA issuer: tcgen05.mma.cta_group::1 kind::f16 M=128 N=128 K=16, 3 per K step, into a double-buffered
//               TMEM accumulator (2 x 128 columns)
//   warps 0-7   epilogue, two warps per TMEM lane quadrant, 64 columns each: dist = sqrtf(2 - 2 clamp(dot, -1, 1)) as
//               nn_match_kernel; row minimum in registers over ascending columns (strict <, so the lowest index wins
//               ties), column minimum by redux.sync.min over the warp's 32 rows (distance bits order like the values) and
//               the lowest row holding it by ballot, merged over the four quadrants in shared memory.  Both minima reach
//               best1 / best2 as 64-bit (distance bits << 32 | index) atomicMin keys: the result does not depend on order.
// nn_select_kernel, one block per pair: mutual test and threshold (fp32, as numpy on the reference's float32 dmat), and an
// order-preserving compaction of the matches.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "tma_map.cuh"
#include <algorithm>

namespace {

constexpr int MT_M = 128;                          // image-1 points per tile (MMA M)
constexpr int MT_N = 128;                          // image-2 points per tile (MMA N)
constexpr int MT_KC = 64;                          // channels per box
constexpr int MT_NKC = 256 / MT_KC;                // 4
constexpr int MT_PLANE_BYTES = MT_M * MT_KC * 2;   // 16 KB: [128 points x 64 channels] bf16
constexpr int MT_BOX_BYTES = 2 * MT_PLANE_BYTES;   // both planes
constexpr int MT_NS = 3;                           // B ring depth
constexpr int MT_THREADS = 320;                    // warps 0-7 epilogue, 8 TMA producer, 9 MMA issuer
constexpr int MT_W_TMA = 8, MT_W_MMA = 9;
constexpr int MT_A_BYTES = MT_NKC * MT_BOX_BYTES;  // 128 KB
constexpr int MT_B_BYTES = MT_NS * MT_BOX_BYTES;   // 96 KB
constexpr int MT_COLKEY_BYTES = MT_N * 8;
constexpr int MT_BAR_BYTES = 256;
constexpr int MT_SMEM = MT_A_BYTES + MT_B_BYTES + MT_COLKEY_BYTES + MT_BAR_BYTES + 1024;  // + alignment slack
static_assert(MT_SMEM <= 227 * 1024, "matcher shared memory");
constexpr uint32_t MT_TMEM_COLS = 2 * MT_N;

struct MatchArgs {
  const unsigned int* counts1;
  const unsigned int* counts2;
  int P, R1, R2;
  int cap1, cap2;  // min(limit, R): the points a pair may use
  unsigned long long* best1;  // [P, R1]
  unsigned long long* best2;  // [P, R2]
};

__device__ __forceinline__ int eff_count(const unsigned int* c, int p, int cap) {
  const unsigned int v = __ldg(c + p);
  return v < (unsigned int)cap ? (int)v : cap;
}

// Walks the flattened item list (pair-major, then row tile, then column tile) over the pairs that hold points.
struct ItemCursor {
  int p, mt, nt, MT, NT, n1, n2;
  __device__ void load(const MatchArgs& a) {
    n1 = eff_count(a.counts1, p, a.cap1);
    n2 = eff_count(a.counts2, p, a.cap2);
    MT = (n1 + MT_M - 1) / MT_M;
    NT = (n2 + MT_N - 1) / MT_N;
    if (MT == 0 || NT == 0) MT = NT = 0;
  }
  __device__ void seek(const MatchArgs& a, long long it) {
    for (p = 0; p < a.P; ++p) {
      load(a);
      const long long k = (long long)MT * NT;
      if (it < k) break;
      it -= k;
    }
    mt = NT ? (int)(it / NT) : 0;
    nt = NT ? (int)(it - (long long)mt * NT) : 0;
  }
  __device__ void next(const MatchArgs& a) {  // only called while items remain
    if (++nt < NT) return;
    nt = 0;
    if (++mt < MT) return;
    mt = 0;
    do { ++p; load(a); } while (MT * NT == 0);
  }
};

__device__ __forceinline__ long long total_items(const MatchArgs& a) {
  long long T = 0;
  for (int p = 0; p < a.P; ++p) {
    const int n1 = eff_count(a.counts1, p, a.cap1), n2 = eff_count(a.counts2, p, a.cap2);
    T += (long long)((n1 + MT_M - 1) / MT_M) * ((n2 + MT_N - 1) / MT_N);
  }
  return T;
}

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }  // the 8 epilogue warps

__global__ void __launch_bounds__(MT_THREADS, 1)
nn_match_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const MatchArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = sA + MT_A_BYTES;
  unsigned long long* colkey = reinterpret_cast<unsigned long long*>(sB + MT_B_BYTES);  // [MT_N] column minima of the item
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + MT_B_BYTES + MT_COLKEY_BYTES);
  uint64_t* a_full = bars;               // [NKC] A box kc has landed
  uint64_t* a_empty = a_full + MT_NKC;   // [NKC] the MMAs of the finished row tile are done with A box kc
  uint64_t* b_full = a_empty + MT_NKC;   // [NS]
  uint64_t* b_empty = b_full + MT_NS;    // [NS]
  uint64_t* t_full = b_empty + MT_NS;    // [2] accumulator complete
  uint64_t* t_empty = t_full + 2;        // [2] the 8 epilogue warps have read it
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long T = total_items(a);
  const long long it0 = T * blockIdx.x / gridDim.x, it1 = T * (blockIdx.x + 1) / gridDim.x;

  if (warp == MT_W_TMA && lane == 0) {
    tc::prefetch_tmap(&tmA);
    tc::prefetch_tmap(&tmB);
  }
  if (warp == MT_W_MMA) {
    if (lane == 0) {
      for (int k = 0; k < MT_NKC; ++k) { tc::mbar_init(a_full + k, 1); tc::mbar_init(a_empty + k, 1); }
      for (int s = 0; s < MT_NS; ++s) { tc::mbar_init(b_full + s, 1); tc::mbar_init(b_empty + s, 1); }
      for (int s = 0; s < 2; ++s) { tc::mbar_init(t_full + s, 1); tc::mbar_init(t_empty + s, 8); }
      tc::fence_barrier_init();
    }
    __syncwarp();
    tc::tmem_alloc(tmem_ptr, MT_TMEM_COLS);
  }
  if (threadIdx.x < MT_N) colkey[threadIdx.x] = ~0ull;
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (it0 < it1) {
    ItemCursor cur;
    cur.seek(a, it0);
    if (warp == MT_W_TMA) {
      // ------------------------------ TMA producer (whole warp loops, one elected lane issues) ------------------------------
      const bool el = tc::elect_one();
      int stage_it = 0, nkeys = 0;
      for (long long it = it0; it < it1; ++it) {
        const bool newkey = it == it0 || cur.nt == 0;
        for (int kc = 0; kc < MT_NKC; ++kc) {
          if (newkey) {
            if (nkeys > 0) tc::mbar_wait(a_empty + kc, (uint32_t)((nkeys - 1) & 1));
            if (el) {
              tc::mbar_expect_tx(a_full + kc, MT_BOX_BYTES);
              tc::tma_load_3d(&tmA, a_full + kc, sA + kc * MT_BOX_BYTES, kc * MT_KC, cur.p * a.R1 + cur.mt * MT_M, 0);
            }
          }
          const int s = stage_it % MT_NS;
          const uint32_t ph = (stage_it / MT_NS) & 1;
          ++stage_it;
          tc::mbar_wait(b_empty + s, ph ^ 1);
          if (el) {
            tc::mbar_expect_tx(b_full + s, MT_BOX_BYTES);
            tc::tma_load_3d(&tmB, b_full + s, sB + s * MT_BOX_BYTES, kc * MT_KC, cur.p * a.R2 + cur.nt * MT_N, 0);
          }
        }
        if (newkey) ++nkeys;
        if (it + 1 < it1) cur.next(a);
      }
      __syncwarp();
    } else if (warp == MT_W_MMA) {
      // ------------------------------ MMA issuer (whole warp loops, one elected lane issues) ------------------------------
      const bool el = tc::elect_one();
      constexpr uint32_t idesc = tc::idesc_bf16_f32(MT_M, MT_N, 0, 0);
      const uint32_t sA_u = tc::smem_u32(sA), sB_u = tc::smem_u32(sB);
      int stage_it = 0, nkeys = 0, tcount = 0;
      for (long long it = it0; it < it1; ++it, ++tcount) {
        const bool newkey = it == it0 || cur.nt == 0;
        if (newkey) ++nkeys;
        const bool last_of_key = it + 1 == it1 || cur.nt == cur.NT - 1;
        const int as = tcount & 1;
        tc::mbar_wait(t_empty + as, ((tcount >> 1) & 1) ^ 1);
        tc::fence_after_sync();
        const uint32_t d_tmem = tmem_base + as * MT_N;
        for (int kc = 0; kc < MT_NKC; ++kc) {
          if (newkey) tc::mbar_wait(a_full + kc, (uint32_t)((nkeys - 1) & 1));
          const int s = stage_it % MT_NS;
          const uint32_t ph = (stage_it / MT_NS) & 1;
          ++stage_it;
          tc::mbar_wait(b_full + s, ph);
          tc::fence_after_sync();
          const uint64_t da_hi = tc::smem_desc_sw128(sA_u + kc * MT_BOX_BYTES, 16, 1024);
          const uint64_t da_lo = tc::smem_desc_sw128(sA_u + kc * MT_BOX_BYTES + MT_PLANE_BYTES, 16, 1024);
          const uint64_t db_hi = tc::smem_desc_sw128(sB_u + s * MT_BOX_BYTES, 16, 1024);
          const uint64_t db_lo = tc::smem_desc_sw128(sB_u + s * MT_BOX_BYTES + MT_PLANE_BYTES, 16, 1024);
          if (el) {
            tc::mma_ss_x4(d_tmem, da_hi, db_hi, idesc, kc > 0 ? 1u : 0u);  // 4 x (M128 N128 K16) over this 64-channel box
            tc::mma_ss_x4(d_tmem, da_lo, db_hi, idesc, 1u);
            tc::mma_ss_x4(d_tmem, da_hi, db_lo, idesc, 1u);
            tc::mma_commit(b_empty + s);
            if (last_of_key) tc::mma_commit(a_empty + kc);
          }
          __syncwarp();
        }
        if (el) tc::mma_commit(t_full + as);
        __syncwarp();
        if (it + 1 < it1) cur.next(a);
      }
    } else {
      // ------------------------------ epilogue warps 0..7 ------------------------------
      const int q = warp & 3, h = warp >> 2;  // TMEM lane quadrant, column half
      uint32_t rbits = ~0u;                   // running row minimum over the row tile's columns seen so far
      int ridx = 0;
      int tcount = 0;
      for (long long it = it0; it < it1; ++it, ++tcount) {
        const bool last_of_key = it + 1 == it1 || cur.nt == cur.NT - 1;
        const int p = cur.p, n1 = cur.n1, n2 = cur.n2, nt = cur.nt;
        const int row = cur.mt * MT_M + q * 32 + lane;
        const bool rowok = row < n1;
        const int as = tcount & 1;
        tc::mbar_wait(t_full + as, (tcount >> 1) & 1);
        tc::fence_after_sync();
        epi_bar();  // the previous item's column keys have been flushed and reset
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          const int cl = h * 64 + ch * 32;  // column of the tile
          const int col0 = nt * MT_N + cl;
          uint32_t v[32];
          tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * MT_N + cl, v);
          tc::tmem_ld_wait();
          uint32_t ckey = ~0u;
          int crow = 0;
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const float dot = fminf(fmaxf(__uint_as_float(v[c]), -1.f), 1.f);
            const uint32_t b = rowok ? __float_as_uint(sqrtf(2.f - 2.f * dot)) : ~0u;
            const bool colok = col0 + c < n2;
            if (colok && b < rbits) { rbits = b; ridx = col0 + c; }
            const uint32_t m = __reduce_min_sync(0xffffffffu, b);
            const uint32_t bal = __ballot_sync(0xffffffffu, b == m);
            if (lane == c) { ckey = m; crow = __ffs(bal) - 1; }
          }
          if (col0 + lane < n2 && ckey != ~0u)
            atomicMin(colkey + cl + lane, ((unsigned long long)ckey << 32) | (unsigned int)(cur.mt * MT_M + q * 32 + crow));
        }
        // all TMEM reads of this stage are complete (wait::ld above): hand the stage back to the MMA warp
        tc::fence_before_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(t_empty + as);
        if (last_of_key) {
          if (rowok && rbits != ~0u)
            atomicMin(a.best1 + (size_t)p * a.R1 + row, ((unsigned long long)rbits << 32) | (unsigned int)ridx);
          rbits = ~0u;
        }
        epi_bar();  // every quadrant has merged its column minima
        if (threadIdx.x < MT_N) {
          const unsigned long long k = colkey[threadIdx.x];
          if (k != ~0ull) atomicMin(a.best2 + (size_t)p * a.R2 + nt * MT_N + threadIdx.x, k);
          colkey[threadIdx.x] = ~0ull;
        }
        if (it + 1 < it1) cur.next(a);
      }
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == MT_W_MMA) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem_base, MT_TMEM_COLS);
  }
}

// One block per pair: keep[i] = dist1[i] < thr && best2[idx1[i]] points back at i, written in increasing i order.
__global__ void __launch_bounds__(256)
nn_select_kernel(const MatchArgs a, float thr, double* __restrict__ matches, unsigned int* __restrict__ nmatch) {
  __shared__ int wcount[8];
  __shared__ int base;
  const int p = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n1 = eff_count(a.counts1, p, a.cap1), n2 = eff_count(a.counts2, p, a.cap2);
  const unsigned long long* b1 = a.best1 + (size_t)p * a.R1;
  const unsigned long long* b2 = a.best2 + (size_t)p * a.R2;
  double* m = matches + (size_t)p * 3 * a.R1;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int i0 = 0; n2 > 0 && i0 < n1; i0 += 256) {
    const int i = i0 + tid;
    bool keep = false;
    int j = 0;
    float dist = 0.f;
    if (i < n1) {
      const unsigned long long k = b1[i];
      j = (int)(k & 0xffffffffull);
      dist = __uint_as_float((unsigned int)(k >> 32));
      keep = k != ~0ull && j < n2 && dist < thr && (int)(b2[j] & 0xffffffffull) == i;
    }
    const unsigned int bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wcount[warp] = __popc(bal);
    __syncthreads();
    int off = base, tot = 0;
    for (int w = 0; w < 8; ++w) {
      if (w < warp) off += wcount[w];
      tot += wcount[w];
    }
    off += __popc(bal & ((1u << lane) - 1u));
    if (keep) {
      m[off] = (double)i;
      m[(size_t)a.R1 + off] = (double)j;
      m[2 * (size_t)a.R1 + off] = (double)dist;
    }
    __syncthreads();
    if (tid == 0) base += tot;
    __syncthreads();
  }
  if (tid == 0) nmatch[p] = (unsigned int)base;
}

}  // namespace

extern "C" size_t ssp_nn_match_batch_ws_bytes(int P, int R1, int R2) {
  return (P > 0 && R1 > 0 && R2 > 0) ? (size_t)P * ((size_t)R1 + (size_t)R2) * 8 : 0;
}

extern "C" int ssp_nn_match_batch(const void* hi1, const void* lo1, int R1, const void* hi2, const void* lo2, int R2,
                                  const unsigned int* counts1, const unsigned int* counts2, int limit, int P,
                                  float nn_thresh, double* matches, unsigned int* nmatch, void* ws, size_t ws_bytes,
                                  void* stream) {
  SSP_REQUIRE(hi1 && lo1 && hi2 && lo2 && counts1 && counts2 && matches && nmatch && ws, "ssp_nn_match_batch: null pointer");
  SSP_REQUIRE(P > 0 && P <= 65535 && R1 > 0 && R2 > 0 && limit > 0, "ssp_nn_match_batch: bad sizes P=%d R1=%d R2=%d limit=%d",
              P, R1, R2, limit);
  SSP_REQUIRE(R1 % 256 == 0 && R2 % 256 == 0, "ssp_nn_match_batch: R1=%d and R2=%d must be multiples of 256", R1, R2);
  SSP_REQUIRE((long long)P * R1 < (1ll << 31) && (long long)P * R2 < (1ll << 31), "ssp_nn_match_batch: P x R too large");
  SSP_REQUIRE(ws_bytes >= ssp_nn_match_batch_ws_bytes(P, R1, R2), "ssp_nn_match_batch: workspace too small");
  SSP_REQUIRE(nn_thresh >= 0.f, "ssp_nn_match_batch: nn_thresh must be non-negative");
  SSP_REQUIRE((((uintptr_t)hi1 | (uintptr_t)lo1 | (uintptr_t)hi2 | (uintptr_t)lo2) & 15) == 0 && ((uintptr_t)ws & 7) == 0,
              "ssp_nn_match_batch: planes must be 16-byte and the workspace 8-byte aligned");
  CUtensorMap mA, mB;
  int rc;
  if ((rc = make_planes_map3(&mA, hi1, lo1, (uint64_t)P * R1, MT_M))) return rc;
  if ((rc = make_planes_map3(&mB, hi2, lo2, (uint64_t)P * R2, MT_N))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  MatchArgs a;
  a.counts1 = counts1; a.counts2 = counts2; a.P = P; a.R1 = R1; a.R2 = R2;
  a.cap1 = std::min(limit, R1); a.cap2 = std::min(limit, R2);
  a.best1 = reinterpret_cast<unsigned long long*>(ws);
  a.best2 = a.best1 + (size_t)P * R1;
  SSP_CUDA_CALL(cudaMemsetAsync(ws, 0xff, ssp_nn_match_batch_ws_bytes(P, R1, R2), st));
  // persistent: one CTA per SM, or fewer when even full pairs hold fewer items
  const long long items = (long long)P * (std::min(limit, R1) / MT_M + 1) * (std::min(limit, R2) / MT_N + 1);
  const int grid = (int)std::min<long long>(items, std::max(1, ssp_num_sms()));
  SSP_CUDA_CALL(cudaFuncSetAttribute(nn_match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MT_SMEM));
  nn_match_tc_kernel<<<grid, MT_THREADS, MT_SMEM, st>>>(mA, mB, a);
  SSP_CUDA_CHECK_LAUNCH("nn_match_tc_kernel");
  nn_select_kernel<<<P, 256, 0, st>>>(a, nn_thresh, matches, nmatch);
  SSP_CUDA_CHECK_LAUNCH("nn_select_kernel");
  return SSP_OK;
}
