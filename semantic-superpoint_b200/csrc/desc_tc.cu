// tcgen05 / TMEM / TMA engine for the dense descriptor loss (sm_100a), CTA-pair (cta_group::2) kernels.
// Reference semantics: utils/utils.py:863-890 (all-pairs dot product + hinge + masks + reductions).
//
// Operands are bf16 K-major planes [B, Nc_pad, 256] produced by desc_pack_kernel: plane "hi" alone
// (mode bf16) or hi + lo with three MMA chains hi*hi + lo*hi + hi*lo (mode bf16x3, ~2^-16 relative
// product error = fp32-grade dot products on the tensor pipe).
//
// Both kernels are persistent over 2-CTA clusters (one per SM pair) and issue M = 256 MMAs over the pair: CTA rank r
// owns rows [128 r, 128 r + 128) of the pair's 256 (its half of A, its half of the accumulator, in ITS tensor memory)
// and supplies HALF of every B tile from its shared memory, so a B tile is fetched from L2 once per pair without
// multicast copies and the B ring holds twice as many stages in the same shared memory.  Rank 0 (the leader) issues every
// tcgen05.mma / tcgen05.commit; TMA bytes of both CTAs are counted on the leader's barriers, commits are multicast.
//
// Forward kernel, work item = (pair b, 256-row tile, 256-column tile; the last column tile is as narrow as Nc needs):
//   warp 8      TMA producer (both CTAs): own 128 A rows (all 256 channels, resident, reloaded chunk by chunk while the
//               last item of the previous row tile still runs), B ring of stages = own half of a [N x 64 ch] chunk, all
//               planes in one 3-D box
//   warp 9      MMA issuer (leader): tcgen05.mma.cta_group::2 kind::f16 M=256 N<=256 K=16 into a double-buffered
//               TMEM accumulator (2 x 256 columns)
//   warps 0-7   epilogue: tcgen05.ld 32x32b, hinge, mask_valid weighting (packed fp32x2 math), running sums and the
//               row-orientation indicator words (sign bits funnel-shifted into place).  No geometry here: the sparse
//               positive pairs are corrected by the pos kernels.  The pair matrix never reaches HBM.
//   The column-orientation indicator words are transposed from the row-orientation ones by blocks of the backward's
//   coefficient launch (desc_pos_coef.cuh).
//
// Backward kernel = indicator GEMM  out[b, d, r] = rowscale[r] * sum_k bit(r,k) * Bp[b, k, d] for the two independent
// jobs (dD and dDw) in one launch, work item = (pair, job, 256-row tile, channel half):
//   warps 0-7   expand 64 indicator bits per row into bf16 {0, 2} (one shift + one and per register; the bit order of
//               the words is chosen for that, DESC_BITPOS) and tcgen05.st them as the A operand into TMEM; warps 0-3 take
//               the even stages, warps 4-7 the odd ones (a single set of four warps was the per-stage critical path:
//               ~130 dependent-issue instructions + the TMEM store round trip per 512 cycles of MMA work)
//   warps 8-15  epilogue of the previous item (double-buffered 128-column accumulators), incl. the sparse
//               positive-pair terms
//   warp 16     TMA producer (both CTAs): ONE 3-D box per stage = [planes x 64 cells x 64 channels] of this CTA's half
//   warp 17     MMA issuer (leader), M=256 N=128 K=16, A from TMEM
#include "desc_common.cuh"
#include "tc_ptx.cuh"
#include "tma_map.cuh"
#include <algorithm>
#include <cstdlib>

// ---- optional timeline trace (build with -DSSP_TRACE, see scripts/trace_desc.py): lane 0 of one warp per role appends
// (clock64 << 8 | tag) records to a per-CTA, per-role slice of the buffer registered with ssp_debug_trace().
#define TRACE_CAP 4096
#ifdef SSP_TRACE
__device__ long long* g_trace_buf = nullptr;
__device__ int g_trace_roles = 0xF;  // bit r: role r records (tracing a role costs it ~40 cycles per record)
#define TR_DECL(role) long long* tr_ = (g_trace_buf && ((g_trace_roles >> (role)) & 1)) ? g_trace_buf + ((size_t)blockIdx.x * 4 + (role)) * TRACE_CAP : nullptr; int trn_ = 0
#define TR_ONLY(cond) do { if (!(cond)) tr_ = nullptr; } while (0)
#define TR(tag) do { if (tr_ && trn_ < TRACE_CAP) tr_[trn_++] = (clock64() << 8) | (long long)(tag); } while (0)
#else
#define TR_DECL(role) do { } while (0)
#define TR_ONLY(cond) do { } while (0)
#define TR(tag) do { } while (0)
#endif

namespace {

constexpr int BM = 128;        // rows per CTA (256 per CTA pair)
constexpr int BN = 256;        // columns per accumulator tile
constexpr int KD = 256;        // descriptor channels (GEMM K of the forward)
constexpr int KC = 64;         // channels per smem chunk = 128 B of bf16 = one swizzle row
constexpr int NKC = KD / KC;   // 4
constexpr int CHUNK_BYTES = BM * KC * 2;  // 16 KB: [128 rows x 64 channels], also one B stage (this CTA's half of a chunk)
constexpr int FWD_THREADS = 320;
constexpr int BAR_BYTES = 1024;  // mbarriers, TMEM pointer

// A B stage = this CTA's half of one 64-channel chunk of a column tile, ALL planes: [P][<=128 cells][64 ch] = P x 16 KB, so that
// the issuing thread pays one barrier wait and one commit per 12 (bf16x3) / 4 (bf16) MMAs.
template <int P> struct FwdCfg {
  static constexpr int A_BYTES = P * NKC * CHUNK_BYTES;
  static constexpr int STAGE_BYTES = P * CHUNK_BYTES;
  static constexpr int NSTAGE = (P == 1) ? 10 : 3;
  static constexpr int B_BYTES = NSTAGE * STAGE_BYTES;
  static constexpr int SMEM = A_BYTES + B_BYTES + BAR_BYTES + 1024;  // + alignment slack
};

__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~(uintptr_t)1023);
}

// One 32-column slice of the accumulator row owned by this thread: negative hinge over every pair (the sparse positive
// pairs are corrected by the pos kernels), mask_valid weighting, row-orientation indicator word.
//   e = mneg - dot (packed), neg = max(-e, 0), su += neg, sw += neg * mv; the indicator of column j is the SIGN of e
//   (dot > mneg), funnel-shifted into bit DESC_BITPOS(j) of the word.  3.5 instructions per pair entry.
template <bool BITS>
__device__ __forceinline__ void epi_chunk(const uint32_t (&v)[32], const float4 (&mq)[8], float mneg, uint64_t& su2,
                                          uint64_t& sw2, uint32_t& rowword) {
  const uint64_t mneg2 = tc::pack2(mneg, mneg);
  uint32_t eb[32];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t e2 = tc::sub2(mneg2, tc::pack2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])));
    float e0, e1;
    tc::unpack2(e2, e0, e1);
    const uint64_t n2 = tc::pack2(fmaxf(-e0, 0.f), fmaxf(-e1, 0.f));
    su2 = tc::add2(su2, n2);
    const float4 m = mq[i >> 1];
    sw2 = tc::fma2(n2, (i & 1) ? tc::pack2(m.z, m.w) : tc::pack2(m.x, m.y), sw2);
    eb[2 * i] = __float_as_uint(e0);
    eb[2 * i + 1] = __float_as_uint(e1);
  }
  if (BITS) {
    uint32_t w = 0;
#pragma unroll
    for (int pos = 31; pos >= 0; --pos) {
      const int j = ((pos & 15) << 1) | (pos >> 4);  // the column whose indicator lives at bit `pos`
      w = __funnelshift_l(eb[j], w, 1);
    }
    rowword = w;
  }
}

// float -> double by bit manipulation (exact for normal numbers and zero; denormals flush to zero, inf / nan kept):
// keeps the epilogue off the FP64 pipe.
__device__ __forceinline__ double f32_to_f64_bits(float f) {
  const uint32_t u = __float_as_uint(f);
  const uint32_t e = (u >> 23) & 0xffu;
  const unsigned long long sign = (unsigned long long)(u & 0x80000000u) << 32;
  unsigned long long d;
  if (e == 0u) d = sign;
  else if (e == 0xffu) d = sign | (0x7ffull << 52) | ((unsigned long long)(u & 0x7fffffu) << 29);
  else d = sign | ((unsigned long long)(e + 896u) << 52) | ((unsigned long long)(u & 0x7fffffu) << 29);
  return __longlong_as_double((long long)d);
}

// Persistent forward kernel.  Work item = (pair b, 256-row tile mp, column tile nt); the flattened item range is split
// evenly over the clusters, items of a cluster are contiguous in nt so the A rows are reloaded only when (b, mp) changes.
// Every epilogue warp keeps its partial sums over all its items (double) and writes ONE pair at the end:
// partials[(cta * 8 + warp) * 2 + {0,1}] -- 1184 entries for the finalize kernel instead of one per item and warp.
// mvbits != NULL ("fold"): the indicator words drop the columns whose mask_valid is 0, so the dD GEMM of the
// backward can run on the unscaled forward planes of Dw (alpha_c = s * mv_c for a binary mask and g_neg = 0).
template <int P, bool BITS>
__global__ void __launch_bounds__(FWD_THREADS, 1)
desc_dense_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmBl, const float* __restrict__ mv_pad, const uint32_t* __restrict__ mvbits, DescGeom g, int n_last,
                         double* __restrict__ partials, uint32_t* __restrict__ bitsR, float* __restrict__ dbgS) {
  using Cfg = FwdCfg<P>;
  constexpr int NSTAGE = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sB = sA + Cfg::A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + Cfg::B_BYTES);
  uint64_t* a_full = bars;              // [NKC]    leader: both CTAs' A chunk kc has landed
  uint64_t* a_empty = a_full + NKC;     // [NKC]    each CTA: the MMAs on A chunk kc of the finished row tile are done
  uint64_t* b_full = a_empty + NKC;     // [NSTAGE] leader: both halves of the stage have landed
  uint64_t* b_empty = b_full + NSTAGE;  // [NSTAGE] each CTA: the MMAs on the stage are done
  uint64_t* t_full = b_empty + NSTAGE;  // [2]      each CTA: accumulator stage complete
  uint64_t* t_empty = t_full + 2;       // [2]      leader: 16 epilogue warps of the pair have drained the stage
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int MP = g.Nc_pad / (2 * BM), NT = g.Nc_pad / BN;  // Nc_pad is a multiple of 256
  const uint32_t cta_rank = tc::cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int ncluster = gridDim.x >> 1, cid = blockIdx.x >> 1;
  const long long T = (long long)g.B * MP * NT;
  const int it0 = (int)(T * cid / ncluster), it1 = (int)(T * (cid + 1) / ncluster);

  if (warp == 8 && lane == 0) {
    tc::prefetch_tmap(&tmA);
    tc::prefetch_tmap(&tmB);
    tc::prefetch_tmap(&tmBl);
  }
  if (warp == 9) {
    if (lane == 0) {
      for (int k = 0; k < NKC; ++k) { tc::mbar_init(a_full + k, 1); tc::mbar_init(a_empty + k, 1); }
      for (int s = 0; s < NSTAGE; ++s) { tc::mbar_init(b_full + s, 1); tc::mbar_init(b_empty + s, 1); }
      for (int s = 0; s < 2; ++s) { tc::mbar_init(t_full + s, 1); tc::mbar_init(t_empty + s, 16); }
      tc::fence_barrier_init();
    }
    __syncwarp();
    tc::tmem_alloc2(tmem_ptr, 512);
  }
  tc::fence_before_sync();
  tc::cluster_sync_all();  // barriers of both CTAs are live before any remote arrive / peer-counted TMA
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 8) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    // The whole warp runs the loop (uniform control flow keeps the TMA / MMA operands in uniform registers; a branch on
    // lane 0 around the loop costs an ELECT / R2UR / BRA.U.ANY waterfall per instruction), one elected lane issues.
    {
      TR_DECL(1);
      TR_ONLY(lane == 0);
      const bool el = tc::elect_one();
      int prev_key = -1, stage_it = 0, nkeys = 0;
      for (int it = it0; it < it1; ++it) {
        const int key = it / NT, nt = it - key * NT;  // key = b * MP + mp
        const int b = key / MP, mp = key - b * MP;
        const int row_base = b * g.Nc_pad;
        const bool newkey = key != prev_key;
        const bool last = nt == NT - 1;
        const int half = (last ? n_last : BN) >> 1;  // B rows (cells) this CTA supplies
        for (int kc = 0; kc < NKC; ++kc) {
          if (newkey) {
            // own 128 rows of A, chunk by chunk: chunk kc is free as soon as the last item of the previous row tile has
            // issued past it, so the reload runs under that item's remaining MMAs
            TR(10);
            if (nkeys > 0) tc::mbar_wait(a_empty + kc, (uint32_t)((nkeys - 1) & 1));
            TR(11);
            if (el) {  // one box: all planes of chunk kc of my 128 rows
              if (leader) tc::mbar_expect_tx(a_full + kc, 2 * P * CHUNK_BYTES);
              tc::tma_load_3d_2sm(&tmA, a_full + kc, sA + kc * P * CHUNK_BYTES, kc * KC, row_base + (2 * mp + (int)cta_rank) * BM, 0);
            }
          }
          {
            const int s = stage_it % NSTAGE;
            const uint32_t ph = (stage_it / NSTAGE) & 1;
            ++stage_it;
            TR(12);
            tc::mbar_wait(b_empty + s, ph ^ 1);
            TR(13);
            if (el) {  // one box: all planes of chunk kc of my half of the tile's columns
              if (leader) tc::mbar_expect_tx(b_full + s, 2 * P * half * KC * 2);
              tc::tma_load_3d_2sm(last ? &tmBl : &tmB, b_full + s, sB + s * Cfg::STAGE_BYTES, kc * KC,
                                  row_base + nt * BN + (int)cta_rank * half, 0);
            }
          }
        }
        if (newkey) { prev_key = key; ++nkeys; }
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------ MMA issuer (leader CTA; whole warp loops, one elected lane issues) ------------------------------
    if (leader) {
      TR_DECL(0);
      TR_ONLY(lane == 0);
      const bool el = tc::elect_one();
      if (tmem_base != 0u) __trap();  // all 512 columns were allocated: the base is column 0, used as a literal below
      const uint32_t sA_u = tc::smem_u32(sA), sB_u = tc::smem_u32(sB);
      int prev_key = -1, stage_it = 0, tcount = 0, nkeys = 0;
      for (int it = it0; it < it1; ++it, ++tcount) {
        const int key = it / NT, nt = it - key * NT;
        const bool newkey = key != prev_key;
        if (newkey) { prev_key = key; ++nkeys; }
        const bool last_of_key = (it + 1 == it1) || ((it + 1) / NT != key);
        const int ncols = nt == NT - 1 ? n_last : BN;
        const uint32_t idesc = tc::idesc_bf16_f32(2 * BM, ncols, 0, 0);
        const int as = tcount & 1;
        const uint32_t aph = (tcount >> 1) & 1;
        TR(2);
        tc::mbar_wait(t_empty + as, aph ^ 1);
        TR(3);
        tc::fence_after_sync();
        const uint32_t d_tmem = as * BN;
        uint32_t first = 1;
        for (int kc = 0; kc < NKC; ++kc) {
          if (newkey) {
            TR(1);
            tc::mbar_wait(a_full + kc, (uint32_t)((nkeys - 1) & 1));
            TR(8);
          }
          {
            const int s = stage_it % NSTAGE;
            const uint32_t ph = (stage_it / NSTAGE) & 1;
            ++stage_it;
            TR(4);
            tc::mbar_wait(b_full + s, ph);
            TR(5);
            tc::fence_after_sync();
            // hi*hi, then (bf16x3) A lo * B hi and A hi * B lo (lo*lo is dropped); plane p of a B stage starts
            // (ncols / 2) * 128 bytes after plane p - 1
            const uint64_t da_hi = tc::smem_desc_sw128(sA_u + (kc * P) * CHUNK_BYTES, 16, 1024);
            const uint64_t db_hi = tc::smem_desc_sw128(sB_u + s * Cfg::STAGE_BYTES, 16, 1024);
            if (el) {
              tc::mma2_ss_x4(d_tmem, da_hi, db_hi, idesc, first ? 0u : 1u);  // 4 x (M256 N K16) over this 64-channel chunk
              if (P == 2) {
                const uint64_t da_lo = tc::smem_desc_sw128(sA_u + (kc * P + 1) * CHUNK_BYTES, 16, 1024);
                const uint64_t db_lo = tc::smem_desc_sw128(sB_u + s * Cfg::STAGE_BYTES + (ncols >> 1) * (KC * 2), 16, 1024);
                tc::mma2_ss_x4(d_tmem, da_lo, db_hi, idesc, 1u);
                tc::mma2_ss_x4(d_tmem, da_hi, db_lo, idesc, 1u);
              }
              tc::mma2_commit_mc(b_empty + s, (uint16_t)0x3);  // both producers: the pair is done with slot s
            }
            first = 0;
            TR(6);
          }
          if (last_of_key && el) tc::mma2_commit_mc(a_empty + kc, (uint16_t)0x3);  // A chunk kc may be replaced in both CTAs
        }
        if (el) tc::mma2_commit_mc(t_full + as, (uint16_t)0x3);  // accumulator tile complete (both CTAs' epilogues)
        __syncwarp();
      }
    }
    __syncwarp();
  } else {
    // ------------------------------ epilogue warps 0..7 (both CTAs) ------------------------------
    const int q = warp & 3, half = warp >> 2;
    const int NW = g.Nc_pad / 32;
    const bool fold = mvbits != nullptr;
    int tcount = 0;
    double su_all = 0.0, sw_all = 0.0;
    TR_DECL(2 + (warp == 7 ? 1 : 0));
    TR_ONLY((warp == 0 || warp == 7) && lane == 0);
    for (int it = it0; it < it1; ++it, ++tcount) {
      const int key = it / NT, nt = it - key * NT;
      const int b = key / MP, mp = key - b * MP;
      const int row_base = b * g.Nc_pad;
      const int m0 = (2 * mp + (int)cta_rank) * BM;
      const int row = m0 + q * 32 + lane;  // row inside the padded pair
      const int ncols = nt == NT - 1 ? n_last : BN;
      const int ch0 = half * 4, ch1 = min((ncols + 31) >> 5, ch0 + 4);  // 32-column chunks of this warp
      const int as = tcount & 1;
      const uint32_t aph = (tcount >> 1) & 1;
      float4 mq[8];
      if (ch0 < ch1) {
        const float4* mvq = reinterpret_cast<const float4*>(mv_pad + (size_t)row_base + nt * BN + ch0 * 32);
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) mq[j4] = __ldg(mvq + j4);
      }
      TR(30);
      tc::mbar_wait(t_full + as, aph);
      TR(31);
      tc::fence_after_sync();
      uint64_t su2 = 0ull, sw2 = 0ull;  // packed fp32 pairs
#pragma unroll 1
      for (int ch = ch0; ch < ch1; ++ch) {
        const int cbase = nt * BN + ch * 32;
        uint32_t v[32];
        tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * BN + ch * 32, v);
        float4 mnext[8];
        if (ch + 1 < ch1) {
          const float4* mvq = reinterpret_cast<const float4*>(mv_pad + (size_t)row_base + cbase + 32);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) mnext[j4] = __ldg(mvq + j4);
        }
        tc::tmem_ld_wait();
        if (ch * 32 + 32 > ncols) {
          // narrow last tile (n_last is a multiple of 16): the upper half of this chunk was not written by the MMA
#pragma unroll
          for (int j = 16; j < 32; ++j) v[j] = 0u;
        }
        uint32_t rowword = 0;
        epi_chunk<BITS>(v, mq, g.mneg, su2, sw2, rowword);
        if (BITS) {
          if (fold) rowword &= __ldg(mvbits + (size_t)b * NW + cbase / 32);
          bitsR[((size_t)b * NW + cbase / 32) * g.Nc_pad + row] = rowword;
        }
        if (dbgS && row < g.Nc) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (cbase + j < g.Nc) dbgS[((size_t)b * g.Nc + row) * g.Nc + cbase + j] = __uint_as_float(v[j]);
        }
        if (ch + 1 < ch1) {
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) mq[j4] = mnext[j4];
        }
      }
      // all TMEM reads of this stage are complete (wait::ld above): hand the stage back to the leader's MMA thread
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive_leader(t_empty + as);
      TR(32);
      float sa, sb, wa, wb;
      tc::unpack2(su2, sa, sb);
      tc::unpack2(sw2, wa, wb);
      su_all += f32_to_f64_bits(sa + sb);  // per-thread, per-item fp32 sums (<= 128 entries) enter a double accumulator
      sw_all += f32_to_f64_bits(wa + wb);
    }
    su_all = warp_sum_d(su_all);
    sw_all = warp_sum_d(sw_all);
    if (lane == 0) {
      const size_t slot = ((size_t)blockIdx.x * 8 + warp) * 2;
      partials[slot] = su_all;
      partials[slot + 1] = sw_all;
    }
  }

  tc::fence_before_sync();
  tc::cluster_sync_all();  // nobody exits while the peer may still arrive on / read from this CTA
  if (warp == 9) {
    tc::fence_after_sync();
    tc::tmem_dealloc2(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// indicator GEMM (backward)
// ------------------------------------------------------------------------------------------------
constexpr int KT = 128;                      // cells (GEMM K) per stage: 8 K=16 steps per plane, i.e. up to 16 MMAs behind ONE pair
                                             // of barrier waits and one commit of the issuing thread (with 64-cell stages that
                                             // thread, not the tensor pipe, set the pace: ~900 cycles per 512 cycles of MMA)
constexpr int BG_PLANE_BYTES = KT * 128;     // one [128 cells x 64 channels] box = 16 KB (this CTA's half of the 128 channels)
constexpr int BG_N = 128;                    // channels per work item (half of the descriptor)
constexpr int BG_THREADS = 576;              // warps 0-7 expanders (two sets), 8-15 epilogue, 16 TMA producer, 17 MMA issuer
constexpr int BG_W_EPI = 8, BG_W_TMA = 16, BG_W_MMA = 17;
constexpr int BG_JOBS = 2;                   // dD and dDw
constexpr int BG_NS = 4;                     // ring depth: TMEM holds 2 x 128 accumulator columns + 4 x 64 columns of A
constexpr int BG_ACOLS = KT / 2;             // TMEM columns of one A stage (two bf16 per column)

constexpr int BG_PF = 4;                     // indicator-word stages in flight per expander set (cp.async groups)
constexpr int BG_WRING_BYTES = 2 * BG_PF * 4 * BM * 4;  // [set][slot][word of the stage][row of the CTA] = 16 KB

template <int P> struct BgCfg {
  static constexpr int STAGE_BYTES = P * BG_PLANE_BYTES;
  static constexpr int SMEM = BG_NS * STAGE_BYTES + BAR_BYTES + BG_WRING_BYTES + 1024;
};

struct BgJob {
  const uint32_t* bits;     // [B, Nc_pad/32, Nc_pad] indicator words of the A operand (rows of this job's output)
  const float* rowscale;    // [B, Nc_pad] or NULL
  const int* plist;         // [B, Nc_pad, DESC_MAXP] positive-pair partners or NULL
  const float* pcoef;       // [B, Nc_pad, DESC_MAXP]
  const uint4* pos_hi;      // packed planes the partners are gathered from
  const uint4* pos_lo;      // NULL: single-pass bf16
  float* out;               // [B, 256, Nc] fp32
};

// Persistent indicator GEMM.  Work item = (pair b, job, 256-row tile mp, channel half dh), round-robin over the clusters
// (at any moment the clusters work on a few consecutive pairs, so their B planes are fetched from HBM once and then hit in
// L2).  The fp32 accumulator is double buffered in TMEM (2 x 128 columns): the epilogue of item i overlaps the main loop
// of item i+1.
template <int P>
__global__ void __launch_bounds__(BG_THREADS, 1)
desc_bits_gemm_tc_kernel(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1, BgJob job0,
                         BgJob job1, int B, int Nc, int Nc_pad) {
  using Cfg = BgCfg<P>;
  constexpr int NS = BG_NS;
  static_assert(256 + BG_ACOLS * NS <= 512, "TMEM A ring does not fit");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NS * Cfg::STAGE_BYTES);
  uint64_t* b_full = bars;          // [NS] leader: both CTAs' B boxes have landed
  uint64_t* a_full = b_full + NS;   // [NS] leader: 8 expander warps of the pair have stored the stage
  uint64_t* s_free = a_full + NS;   // [NS] each CTA: the MMAs on the stage are done
  uint64_t* d_full = s_free + NS;   // [2]  each CTA: accumulator complete
  uint64_t* d_empty = d_full + 2;   // [2]  leader: 16 epilogue warps of the pair have drained it
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(d_empty + 2);
  uint32_t* wring = reinterpret_cast<uint32_t*>(smem + NS * Cfg::STAGE_BYTES + BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int MP = Nc_pad / (2 * BM), NK = (Nc + KT - 1) / KT, NW = Nc_pad / 32;
  const int NKS = (Nc + 15) / 16;  // K=16 steps that hold real cells: the last stage issues only its share of them
  const uint32_t cta_rank = tc::cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int ncluster = gridDim.x >> 1, cid = blockIdx.x >> 1;
  const int T = B * BG_JOBS * MP * 2;
  constexpr uint32_t A_COL0 = 256;  // TMEM: accumulators at columns [0,128) and [128,256), then NS x 64 columns of A

  // item -> (b, job, mp, dh)
  auto decode = [&](int it, int& b, int& jb, int& mp, int& dh) {
    dh = it & 1;
    int t = it >> 1;
    mp = t % MP;
    t /= MP;
    jb = t % BG_JOBS;
    b = t / BG_JOBS;
  };

  if (warp == BG_W_TMA && lane == 0) {
    tc::prefetch_tmap(&tm0);
    tc::prefetch_tmap(&tm1);
  }
  if (warp == BG_W_MMA) {
    if (lane == 0) {
      for (int s = 0; s < NS; ++s) { tc::mbar_init(b_full + s, 1); tc::mbar_init(a_full + s, 8); tc::mbar_init(s_free + s, 1); }
      for (int s = 0; s < 2; ++s) { tc::mbar_init(d_full + s, 1); tc::mbar_init(d_empty + s, 16); }
      tc::fence_barrier_init();
    }
    __syncwarp();
    tc::tmem_alloc2(tmem_ptr, 512);
  }
  tc::fence_before_sync();
  tc::cluster_sync_all();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == BG_W_TMA) {
    // ------------------------------ TMA producer (both CTAs; whole warp loops, one elected lane issues) ------------------------------
    {
      TR_DECL(1);
      TR_ONLY(lane == 0);
      const bool el = tc::elect_one();
      int st_it = 0;
      for (int it = cid; it < T; it += ncluster) {
        int b, jb, mp, dh;
        decode(it, b, jb, mp, dh);
        const CUtensorMap* m = jb ? &tm1 : &tm0;
        for (int kc = 0; kc < NK; ++kc, ++st_it) {
          const int s = st_it % NS;
          const uint32_t ph = (st_it / NS) & 1;
          TR(12);
          tc::mbar_wait(s_free + s, ph ^ 1);
          TR(13);
          if (el) {
            if (leader) tc::mbar_expect_tx(b_full + s, 2 * Cfg::STAGE_BYTES);
            // one box: [P planes x 128 cells x my 64 of the item's 128 channels]
            tc::tma_load_3d_2sm(m, b_full + s, smem + s * Cfg::STAGE_BYTES, dh * BG_N + (int)cta_rank * 64, b * Nc_pad + kc * KT, 0);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == BG_W_MMA) {
    // ------------------------------ MMA issuer (leader CTA; whole warp loops, one elected lane issues) ------------------------------
    if (leader) {
      TR_DECL(0);
      TR_ONLY(lane == 0);
      const bool el = tc::elect_one();
      if (tmem_base != 0u) __trap();  // all 512 columns were allocated: the base is column 0, used as a literal below
      constexpr uint32_t idesc = tc::idesc_bf16_f32(2 * BM, BG_N, 0, 1);  // A K-major (TMEM), B MN-major
      const uint32_t smem_u = tc::smem_u32(smem);
      int st_it = 0, tcount = 0;
      for (int it = cid; it < T; it += ncluster, ++tcount) {
        const int as = tcount & 1;
        const uint32_t aph = (tcount >> 1) & 1;
        TR(2);
        tc::mbar_wait(d_empty + as, aph ^ 1);
        TR(3);
        tc::fence_after_sync();
        const uint32_t d_tmem = as * BG_N;
        uint32_t first = 1;
        for (int kc = 0; kc < NK; ++kc, ++st_it) {
          const int s = st_it % NS;
          const uint32_t ph = (st_it / NS) & 1;
          TR(4);
          tc::mbar_wait(b_full + s, ph);
          TR(5);
          tc::mbar_wait(a_full + s, ph);
          TR(7);
          tc::fence_after_sync();
          const int nks = min(KT / 16, NKS - kc * (KT / 16));  // K=16 steps of this stage that hold real cells
          for (int p = 0; p < P; ++p) {
            // per K=16 step: 16 cells = two 8-row groups (SBO 1024 B, +2048 B = 128 descriptor units per step); each CTA
            // supplies one 64-channel swizzle atom of the 128 channels; A advances 8 TMEM columns per step
            const uint64_t db = tc::smem_desc_sw128(smem_u + s * Cfg::STAGE_BYTES + p * BG_PLANE_BYTES, BG_PLANE_BYTES, 1024);
            for (int j = 0; j < nks; ++j) {
              if (el) tc::mma2_ts(d_tmem, A_COL0 + s * BG_ACOLS + 8 * j, db + (uint64_t)(128 * j), idesc, first ? 0u : 1u);
              first = 0;
            }
          }
          if (el) tc::mma2_commit_mc(s_free + s, (uint16_t)0x3);
          TR(6);
        }
        if (el) tc::mma2_commit_mc(d_full + as, (uint16_t)0x3);
        __syncwarp();
      }
    }
    __syncwarp();
  } else if (warp < BG_W_EPI) {
    // ------------------------------ expanders (both CTAs): indicator bits -> bf16 A operand in TMEM ------------------------------
    const int q = warp & 3, set = warp >> 2;  // TMEM lane quadrant; set 0 expands the even stages, set 1 the odd ones
    TR_DECL(2);
    TR_ONLY(warp == 0 && lane == 0);
    // one ring stage: the 128 indicator bits (four words) of this row become 64 TMEM columns of bf16 pairs.  Bit i of a word
    // is cell 2i, bit 16+i is cell 2i+1 (DESC_BITPOS), so column i of a word is ONE shift and ONE and:
    // (w << (14 - i)) & 0x40004000 -- bf16 0x4000 = 2.0; the epilogue multiplies by 0.5.
    auto expand_words = [&](uint32_t w0, uint32_t w1, uint32_t (&r)[32]) {
#pragma unroll
      for (int i = 0; i < 15; ++i) {
        r[i] = (w0 << (14 - i)) & 0x40004000u;
        r[16 + i] = (w1 << (14 - i)) & 0x40004000u;
      }
      r[15] = (w0 >> 1) & 0x40004000u;
      r[31] = (w1 >> 1) & 0x40004000u;
    };
    auto expand_stage = [&](int st_it, const uint32_t (&w)[4]) {
      const int s = st_it % NS;
      const uint32_t ph = (st_it / NS) & 1;
      uint32_t r[32];
      expand_words(w[0], w[1], r);
      TR(20);
      tc::mbar_wait(s_free + s, ph ^ 1);
      TR(21);
      tc::fence_after_sync();
      const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + A_COL0 + s * BG_ACOLS;
      tc::tmem_st32(t0, r);
      expand_words(w[2], w[3], r);
      tc::tmem_st32(t0 + 32, r);
      tc::tmem_st_wait();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive_leader(a_full + s);
      TR(23);
    };
    // The indicator words run PF of this set's stages ahead of their use over the FLAT stage sequence of all items of this
    // cluster, so neither the L2 latency inside an item nor the start of a new item is exposed.  They travel through shared
    // memory with cp.async (one commit group per stage, every thread copies and later reads only ITS OWN four words, so no
    // barrier is involved): as register prefetches the loads of different stages shared the warp's six scoreboards, and
    // waiting for the oldest stage also waited for the one just issued -- ncu showed the expanders stalled on the first use
    // of a word for a full L2 round trip per stage, which made them, not the tensor pipe, the pace of the kernel.
    constexpr int PF = BG_PF;
    uint32_t* myring = wring + (size_t)set * PF * 4 * BM + (q * 32 + lane);  // + (slot * 4 + word) * BM
    int itB = cid, kcB = set;  // fetch cursor (stage `set` of the first item)
    const uint32_t* pB = nullptr;
    bool newitem = true;
    auto fetch = [&](int slot) {
      while (itB < T && kcB >= NK) { kcB -= NK; itB += ncluster; newitem = true; }  // NK may be 1 (tiny inputs)
      if (itB < T) {
        if (newitem) {
          int b, jb, mp, dh;
          decode(itB, b, jb, mp, dh);
          const int row = (2 * mp + (int)cta_rank) * BM + q * 32 + lane;
          pB = (jb ? job1.bits : job0.bits) + (size_t)b * NW * Nc_pad + row;
          newitem = false;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) tc::cp_async4(myring + (slot * 4 + u) * BM, pB + (size_t)(4 * kcB + u) * Nc_pad);
        kcB += 2;
      }
      tc::cp_async_commit();  // an empty group when the items are exhausted: the group count stays in step with the slots
    };
#pragma unroll
    for (int u = 0; u < PF; ++u) fetch(u);
    const int nitems = cid < T ? (T - cid + ncluster - 1) / ncluster : 0;
    const int total = nitems * NK;  // global stage count of this cluster; this set owns g = set, set + 2, ...
    for (int g0 = set; g0 < total; g0 += 2 * PF) {
#pragma unroll
      for (int u = 0; u < PF; ++u) {
        if (g0 + 2 * u < total) {
          tc::cp_async_wait<PF - 1>();  // the oldest outstanding group = slot u
          uint32_t w[4];
#pragma unroll
          for (int v = 0; v < 4; ++v) w[v] = myring[(u * 4 + v) * BM];
          expand_stage(g0 + 2 * u, w);
          fetch(u);
        }
      }
    }
    tc::cp_async_wait<0>();
  } else {
    // ------------------------------ epilogue warps 8..15 (both CTAs) ------------------------------
    // two warps per TMEM lane quadrant, each draining two of the four 32-column chunks of the accumulator
    const int q = warp & 3, chalf = (warp - BG_W_EPI) >> 2;
    int tcount = 0;
    TR_DECL(3);
    TR_ONLY(warp == BG_W_EPI && lane == 0);
    for (int it = cid; it < T; it += ncluster, ++tcount) {
      int b, jb, mp, dh;
      decode(it, b, jb, mp, dh);
      const BgJob& J = jb ? job1 : job0;
      const int row = (2 * mp + (int)cta_rank) * BM + q * 32 + lane;
      const bool row_ok = row < Nc;
      float rs = 0.5f;  // the A operand holds 2.0 for a set indicator
      if (J.rowscale && row_ok) rs *= J.rowscale[(size_t)b * Nc_pad + row];
      // sparse positive pairs of this row (and removal of their negative term, see desc_pos_coef_kernel): their
      // gathers hide behind the next item's main loop because this epilogue runs on its own warps
      const int* pl = J.plist ? J.plist + ((size_t)b * Nc_pad + row) * DESC_MAXP : nullptr;
      const float* pcf = J.plist ? J.pcoef + ((size_t)b * Nc_pad + row) * DESC_MAXP : nullptr;
      int npos = 0;
      if (pl && row_ok) {
#pragma unroll
        for (int n = 0; n < DESC_MAXP; ++n)
          if (pl[n] >= 0) npos = n + 1;
      }
      const int nmax = __reduce_max_sync(0xffffffffu, npos);
      const int as = tcount & 1;
      const uint32_t aph = (tcount >> 1) & 1;
      TR(30);
      tc::mbar_wait(d_full + as, aph);
      TR(31);
      tc::fence_after_sync();
      // adds the positive-pair terms of partner list entry n to the 32 channels of chunk ch held in val[]
      auto add_partner = [&](int n, int ch, float (&val)[32]) {
        int pc = n < npos ? pl[n] : -1;
        if (pc < 0) return;
        float pf = pcf[n];
        // partner descriptor from the packed planes: the 32 channels of this chunk are 64 contiguous bytes per
        // plane (4 x 16 B per lane, every fetched sector fully used)
        const size_t o = (((size_t)b * Nc_pad + pc) * KD + dh * BG_N + ch * 32) >> 3;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint4 h = __ldg(J.pos_hi + o + u);
          const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
          uint32_t lw[4] = {0u, 0u, 0u, 0u};
          if (J.pos_lo) {
            const uint4 l = __ldg(J.pos_lo + o + u);
            lw[0] = l.x; lw[1] = l.y; lw[2] = l.z; lw[3] = l.w;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float e0 = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
            float e1 = __uint_as_float(hw[i] & 0xffff0000u) + __uint_as_float(lw[i] & 0xffff0000u);
            val[u * 8 + 2 * i] = fmaf(pf, e0, val[u * 8 + 2 * i]);
            val[u * 8 + 2 * i + 1] = fmaf(pf, e1, val[u * 8 + 2 * i + 1]);
          }
        }
      };
#pragma unroll 1
      for (int ch = chalf * 2; ch < chalf * 2 + 2; ++ch) {
        uint32_t v[32];
        tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * BG_N + ch * 32, v);
        tc::tmem_ld_wait();
        if (row_ok) {
          float val[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) val[j] = __uint_as_float(v[j]) * rs;
#pragma unroll 1
          for (int n = 0; n < nmax; ++n) add_partner(n, ch, val);
          float* o = J.out + ((size_t)b * KD + dh * BG_N + ch * 32) * Nc + row;
#pragma unroll
          for (int j = 0; j < 32; ++j) o[(size_t)j * Nc] = val[j];
        }
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive_leader(d_empty + as);
      TR(32);
    }
  }

  tc::fence_before_sync();
  tc::cluster_sync_all();
  if (warp == BG_W_MMA) {
    tc::fence_after_sync();
    tc::tmem_dealloc2(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// launch with thread-block clusters of 2 along x
template <typename... KArgs, typename... Args>
int launch_cluster2(void (*kernel)(KArgs...), int grid, int block, int smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
  if (e != cudaSuccess) { ssp_set_error("cluster launch failed: %s", cudaGetErrorString(e)); return (int)e; }
  return SSP_OK;
}

template <typename K>
int set_smem(K kernel, int bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) { ssp_set_error("cudaFuncSetAttribute(%d B smem) failed: %s", bytes, cudaGetErrorString(e)); return (int)e; }
  return SSP_OK;
}

}  // namespace

// Profiling aid: registers a device buffer of n_cta * 4 * TRACE_CAP int64 records for the timeline trace of the two tensor-core
// kernels (library built with -DSSP_TRACE only; otherwise SSP_EUNSUPPORTED).  NULL switches tracing off.
extern "C" int ssp_debug_trace(void* buf) {
#ifdef SSP_TRACE
  long long* p = reinterpret_cast<long long*>(buf);
  SSP_CUDA_CALL(cudaMemcpyToSymbol(g_trace_buf, &p, sizeof(p)));
  const char* e = getenv("SSP_TRACE_ROLES");  // bit mask of the roles that record (default all four)
  int roles = e ? atoi(e) : 0xF;
  SSP_CUDA_CALL(cudaMemcpyToSymbol(g_trace_roles, &roles, sizeof(roles)));
  return SSP_OK;
#else
  (void)buf;
  ssp_set_error("ssp_debug_trace: library built without -DSSP_TRACE");
  return SSP_EUNSUPPORTED;
#endif
}
extern "C" int ssp_debug_trace_cap(void) { return TRACE_CAP; }

// partial-sum slots of the forward kernel: one per (CTA, epilogue warp) of the persistent grid
extern "C" int ssp_desc_dense_tc_nblocks(int B, int Nc) {
  int ncp = desc_nc_pad(Nc);
  long long items = (long long)B * (ncp / (2 * BM)) * (ncp / BN);
  int nclusters = (int)std::min<long long>(items, std::max(1, ssp_num_sms() / 2));
  return 2 * nclusters * 8;
}

// Ahi/Alo: packed planes of `descriptors`, Bhi/Blo: packed planes of `descriptors_warped` ([B, Nc_pad, 256] bf16).
// Alo == Blo == NULL selects single-pass bf16; otherwise bf16x3.  bitsR (optional) receives the row-orientation indicator
// words (their transpose bitsC comes from ssp_desc_pos_coef).  mvbits (optional, [B, Nc_pad/32] words of mask_valid != 0 in
// DESC_BITPOS order, from ssp_desc_pack2_geometry): the indicator words drop the columns whose mask_valid is 0 ("fold").
extern "C" int ssp_desc_dense_fwd_tc(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo,
                                     const float* mv_pad, const uint32_t* mvbits, int B, int Hc, int Wc, float mneg,
                                     double* partials, uint32_t* bitsR, float* dbgS, void* stream) {
  SSP_REQUIRE(Ahi && Bhi && mv_pad && partials, "ssp_desc_dense_fwd_tc: null pointer");
  SSP_REQUIRE((Alo == nullptr) == (Blo == nullptr), "ssp_desc_dense_fwd_tc: lo planes must both be given or both null");
  SSP_REQUIRE(B > 0 && B <= 65535 && Hc > 0 && Wc > 0, "ssp_desc_dense_fwd_tc: bad sizes");
  SSP_REQUIRE(mneg > 0.f, "ssp_desc_dense_fwd_tc: margin_neg must be > 0 (zero padding relies on it)");
  SSP_REQUIRE((((uintptr_t)Ahi | (uintptr_t)Bhi | (uintptr_t)Alo | (uintptr_t)Blo | (uintptr_t)mv_pad) & 15) == 0,
              "ssp_desc_dense_fwd_tc: operands must be 16-byte aligned");
  DescGeom g;
  g.B = B; g.Hc = Hc; g.Wc = Wc; g.Nc = Hc * Wc; g.Nc_pad = desc_nc_pad(g.Nc); g.Dch = KD;
  g.cell = 0; g.dist = 0.f; g.lamda = 0.f; g.mpos = 0.f; g.mneg = mneg;
  const int NT = g.Nc_pad / BN;
  const int n_last = ((g.Nc - (NT - 1) * BN) + 15) / 16 * 16;  // width of the last column tile: 16..256, multiple of 16
  uint64_t rows = (uint64_t)B * g.Nc_pad;
  CUtensorMap mA, mB, mL;
  int rc;
  if ((rc = make_planes_map3(&mA, Ahi, Alo, rows, BM))) return rc;
  if ((rc = make_planes_map3(&mB, Bhi, Blo, rows, BN / 2))) return rc;  // each CTA of a pair supplies half of the tile's columns
  if ((rc = make_planes_map3(&mL, Bhi, Blo, rows, n_last / 2))) return rc;
  // persistent: one 2-CTA cluster per SM pair (or fewer when there is less work)
  long long items = (long long)B * (g.Nc_pad / (2 * BM)) * NT;
  int nclusters = (int)std::min<long long>(items, std::max(1, ssp_num_sms() / 2));
  int grid = 2 * nclusters;
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_FWD(PP, BB)                                                                                       \
  do {                                                                                                           \
    if ((rc = set_smem(desc_dense_fwd_tc_kernel<PP, BB>, FwdCfg<PP>::SMEM))) return rc;                          \
    if ((rc = launch_cluster2(desc_dense_fwd_tc_kernel<PP, BB>, grid, FWD_THREADS, FwdCfg<PP>::SMEM, st, mA, mB, mL,         \
                              mv_pad, mvbits, g, n_last, partials, bitsR, dbgS))) return rc;                     \
  } while (0)
  if (Alo) { if (bitsR) LAUNCH_FWD(2, true); else LAUNCH_FWD(2, false); }
  else     { if (bitsR) LAUNCH_FWD(1, true); else LAUNCH_FWD(1, false); }
#undef LAUNCH_FWD
  SSP_CUDA_CHECK_LAUNCH("desc_dense_fwd_tc_kernel");
  return SSP_OK;
}

// Both indicator GEMMs of the backward in ONE launch (job 0: dD, job 1: dDw; Blo / pos_lo NULL: single-pass bf16 engine):
//   out[b, d, r] = rowscale[b, r] * sum_k bit(r, k) * (Bhi + Blo)[b, k, d]      (out is [B, 256, Nc] fp32)
//                  + sum_n pcoef[b, r, n] * (pos_hi + pos_lo)[b, plist[b, r, n], d]   (sparse positive pairs; plist may be NULL)
// Two jobs per launch give 2x the work items, so the persistent clusters end within one item of each other (4.3 items per
// cluster for one job at B = 32, 8.6 for two).
extern "C" int ssp_desc_bits_gemm_tc_pair(const uint32_t* bits0, const void* Bhi0, const void* Blo0, const float* rowscale0,
                                          const int* plist0, const float* pcoef0, const void* pos_hi0, const void* pos_lo0,
                                          float* out0, const uint32_t* bits1, const void* Bhi1, const void* Blo1,
                                          const float* rowscale1, const int* plist1, const float* pcoef1, const void* pos_hi1,
                                          const void* pos_lo1, float* out1, int B, int Nc, void* stream) {
  SSP_REQUIRE(B > 0 && Nc > 0, "ssp_desc_bits_gemm_tc_pair: bad sizes");
  SSP_REQUIRE(bits0 && Bhi0 && out0 && bits1 && Bhi1 && out1, "ssp_desc_bits_gemm_tc_pair: null pointer");
  SSP_REQUIRE((!plist0 || (pcoef0 && pos_hi0)) && (!plist1 || (pcoef1 && pos_hi1)),
              "ssp_desc_bits_gemm_tc_pair: plist needs pcoef and the partner planes");
  SSP_REQUIRE((((uintptr_t)Bhi0 | (uintptr_t)Blo0 | (uintptr_t)pos_hi0 | (uintptr_t)pos_lo0 | (uintptr_t)Bhi1 | (uintptr_t)Blo1 |
                (uintptr_t)pos_hi1 | (uintptr_t)pos_lo1) & 15) == 0,
              "ssp_desc_bits_gemm_tc_pair: operands must be 16-byte aligned");
  SSP_REQUIRE((Blo0 == nullptr) == (Blo1 == nullptr), "ssp_desc_bits_gemm_tc_pair: both jobs must use the same engine (lo planes)");
  const int Nc_pad = desc_nc_pad(Nc);
  const uint64_t rows = (uint64_t)B * Nc_pad;
  CUtensorMap m0, m1;
  int rc;
  if ((rc = make_planes_map3(&m0, Bhi0, Blo0, rows, KT))) return rc;
  if ((rc = make_planes_map3(&m1, Bhi1, Blo1, rows, KT))) return rc;
  const BgJob j0 = {bits0, rowscale0, plist0, pcoef0, (const uint4*)pos_hi0, (const uint4*)pos_lo0, out0};
  const BgJob j1 = {bits1, rowscale1, plist1, pcoef1, (const uint4*)pos_hi1, (const uint4*)pos_lo1, out1};
  long long items = (long long)B * BG_JOBS * (Nc_pad / (2 * BM)) * 2;
  int nclusters = (int)std::min<long long>(items, std::max(1, ssp_num_sms() / 2));
  int grid = 2 * nclusters;
  cudaStream_t st = (cudaStream_t)stream;
  if (Blo0) {
    if ((rc = set_smem(desc_bits_gemm_tc_kernel<2>, BgCfg<2>::SMEM))) return rc;
    if ((rc = launch_cluster2(desc_bits_gemm_tc_kernel<2>, grid, BG_THREADS, BgCfg<2>::SMEM, st, m0, m1, j0, j1, B, Nc, Nc_pad)))
      return rc;
  } else {
    if ((rc = set_smem(desc_bits_gemm_tc_kernel<1>, BgCfg<1>::SMEM))) return rc;
    if ((rc = launch_cluster2(desc_bits_gemm_tc_kernel<1>, grid, BG_THREADS, BgCfg<1>::SMEM, st, m0, m1, j0, j1, B, Nc, Nc_pad)))
      return rc;
  }
  SSP_CUDA_CHECK_LAUNCH("desc_bits_gemm_tc_kernel");
  return SSP_OK;
}
