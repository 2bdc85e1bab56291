// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma /
// commit / ld / st / fences) and UMMA descriptor construction.  Bit layouts follow the PTX ISA
// "tcgen05 matrix descriptors" (same fields as cute::UMMA::SmemDescriptor / InstrDescriptor).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------- cp.async (per-thread asynchronous copies tracked by commit groups, not by scoreboards) ----------------
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---------------- TMA ----------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// 2-D tiled load global -> shared, completes `bytes` on the mbarrier
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}

// 3-D tiled load global -> shared (this CTA), completes `bytes` on the mbarrier
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* dst, int x, int y, int z) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z)
      : "memory");
}

// same, delivered to the same smem / mbarrier offsets of every CTA in `cta_mask` of the cluster (L2 read once)
__device__ __forceinline__ void tma_load_2d_mc(const CUtensorMap* m, uint64_t* bar, void* dst, int x, int y, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(x), "r"(y), "h"(cta_mask)
      : "memory");
}

// one lane of the (converged) warp: used to predicate single-thread instructions inside warp-uniform loops, so that their
// operands stay in uniform registers (a branch on lane == 0 around the whole loop makes ptxas emit an ELECT / R2UR /
// BRA.U.ANY waterfall per tcgen05.mma: ~100 cycles of issue per instruction, measured)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------- clusters ----------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------- tcgen05 ----------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]      (kind::f16: bf16/f16 inputs, fp32 accumulate)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Four K=16 steps of one 64-element (128 B) swizzled K chunk in ONE asm block: the descriptors advance by
// 2 x 16-byte units (32 B along K) per MMA.  One block per chunk keeps the single-thread issue path short
// (the register -> uniform-register moves happen once per block, not once per MMA).
__device__ __forceinline__ void mma_ss_x4(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, pt;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      "add.s64 a1, %1, 2;\n\tadd.s64 a2, %1, 4;\n\tadd.s64 a3, %1, 6;\n\t"
      "add.s64 b1, %2, 2;\n\tadd.s64 b2, %2, 4;\n\tadd.s64 b3, %2, 6;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, pt;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, pt;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, pt;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Four K=16 steps with A in TMEM (8 columns per step) and an MN-major B tile (16 rows = 2048 B = 128 units per step)
__device__ __forceinline__ void mma_ts_x4(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, pt;\n\t.reg .b64 b1, b2, b3;\n\t.reg .b32 a1, a2, a3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      "add.s32 a1, %1, 8;\n\tadd.s32 a2, %1, 16;\n\tadd.s32 a3, %1, 24;\n\t"
      "add.s64 b1, %2, 128;\n\tadd.s64 b2, %2, 256;\n\tadd.s64 b3, %2, 384;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a1], b1, %3, pt;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a2], b2, %3, pt;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [a3], b3, %3, pt;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// same, arriving on the barrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void mma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive 32-bit columns; thread t of the warp reads lane (base+t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM, same shape
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// =====================================================================================================
// cta_group::2 (CTA pair) forms.  The pair = the two CTAs of a 2-CTA cluster; rank 0 is the leader: it issues every
// tcgen05.mma / tcgen05.commit and owns the barriers that collect both CTAs' TMA bytes and arrivals.  A shared::cta
// address with bit 24 cleared names the same offset in the leader's shared memory (cute::Sm100MmaPeerBitMask).
// =====================================================================================================
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {  // one whole warp of EACH CTA, same dst offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {  // one whole warp of EACH CTA
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive on the barrier at this offset in the LEADER CTA (callable from either CTA of the pair).  Default semantics, as
// cutlass::arch::umma_arrive_2x1SM_sm0: an explicit .release.cluster would put MEMBAR.ALL.GPU + ERRBAR in front of every
// arrive (measured: it serialised the expander warps behind their own indicator-word prefetches, 2.4 k cycles per stage).
// What the arrive publishes is tensor memory, which tcgen05.wait::st / tcgen05.fence::before_thread_sync order.
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
// TMA loads of a CTA pair: data lands in THIS CTA's shared memory, the bytes are counted on the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* m, uint64_t* bar, void* dst, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & kPeerBitMask), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(const CUtensorMap* m, uint64_t* bar, void* dst, int x, int y, int z) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & kPeerBitMask), "r"(x), "r"(y), "r"(z)
      : "memory");
}
// Four K=16 steps of one 64-element swizzled K chunk, M = 256 over the CTA pair (A and B from shared memory)
__device__ __forceinline__ void mma2_ss_x4(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, pt;\n\t.reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      "add.s64 a1, %1, 2;\n\tadd.s64 a2, %1, 4;\n\tadd.s64 a3, %1, 6;\n\t"
      "add.s64 b1, %2, 2;\n\tadd.s64 b2, %2, 4;\n\tadd.s64 b3, %2, 6;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], a1, b1, %3, pt;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], a2, b2, %3, pt;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], a3, b3, %3, pt;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Four K=16 steps with A in TMEM (8 columns per step, same address in both CTAs) and an MN-major B tile
// (16 rows = 2048 B = 128 descriptor units per step), M = 256 over the CTA pair
__device__ __forceinline__ void mma2_ts_x4(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, pt;\n\t.reg .b64 b1, b2, b3;\n\t.reg .b32 a1, a2, a3;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 pt, 0, 0;\n\t"
      "add.s32 a1, %1, 8;\n\tadd.s32 a2, %1, 16;\n\tadd.s32 a3, %1, 24;\n\t"
      "add.s64 b1, %2, 128;\n\tadd.s64 b2, %2, 256;\n\tadd.s64 b3, %2, 384;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a1], b1, %3, pt;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a2], b2, %3, pt;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [a3], b3, %3, pt;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// single K=16 step, A in TMEM (pair MMA)
__device__ __forceinline__ void mma2_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all previously issued MMAs of the pair have completed) on the barrier at this offset in the CTAs of `cta_mask`
__device__ __forceinline__ void mma2_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
// same, leader's barrier only
__device__ __forceinline__ void mma2_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// registers -> TMEM, 32 lanes x 16 consecutive columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ---------------- packed fp32x2 arithmetic (FADD2 / FFMA2) ----------------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

// ---------------- descriptors ----------------
// Shared-memory matrix descriptor, SWIZZLE_128B, 16-bit elements.
//  K-major  tile [rows x 64 elem]: rows 128 B apart, 8-row groups SBO = 1024 B apart (LBO unused = 1).
//  MN-major tile [k rows x 64 elem] blocks: 8-k groups SBO = 1024 B apart, next 64 MN elements LBO bytes on.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulate.
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                           // c_format = F32
         | (1u << 7)                         // a_format = BF16
         | (1u << 10)                        // b_format = BF16
         | ((uint32_t)a_mn_major << 15)      // A major-ness (0 = K)
         | ((uint32_t)b_mn_major << 16)      // B major-ness (0 = K)
         | ((uint32_t)(N >> 3) << 17)        // n_dim
         | ((uint32_t)(M >> 4) << 24);       // m_dim
}

}  // namespace tc
