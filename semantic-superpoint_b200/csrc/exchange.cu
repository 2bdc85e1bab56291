// Multi-GPU exchange of the global-batch normalisers (SURVEY 8e) as ONE kernel over peer memory.
//
// Reference semantics: both losses divide by whole-batch quantities --
//   detector_loss   sum(mask) + 1e-5                       Train_model_heatmap_all.py:178
//   descriptor_loss B * (sum(mask_valid) + 1) * Hc * Wc     utils/utils.py:886-887
//   sem_loss        number of counted pixels               Train_model_heatmap_all.py:181-193
// so a batch sharded over G GPUs needs the sum over ranks of <= 13 scalars per step and nothing else.  Each rank owns a
// small exchange buffer (cudaMalloc, exported with cudaIpc so that the other processes of the node map it over
// NVLink / NVSwitch peer access).  The kernel (one warp)
//   1. PUSHES its 16-float payload into slot [parity][rank] of every rank's buffer (4 x 16-byte peer stores),
//      system fence, then a release store of the sequence number into flag [parity][rank] of that buffer;
//   2. spins (acquire loads of LOCAL memory only) until the flags of all ranks carry this sequence number;
//   3. adds the slots in rank order (deterministic, identical on every rank) and rewrites the loss triples / the
//      descriptor out8 in place with the global-batch values, exactly the fix-ups the reference formulas imply.
// Slots are double buffered by the parity of the sequence number: a rank can only be one exchange ahead of a peer
// (it needs the peer's flag of exchange n to finish n), so slot n+1 never overwrites data a slow peer still reads.
// No NCCL call, no host synchronisation; capturable in a CUDA graph (the sequence counter lives in device memory).
#include "common.cuh"
#include <string.h>

#define XCHG_MAXR 16  // ranks per node
#define XCHG_NV 16    // floats per payload

struct XchgBuf {
  unsigned int seq;                       // exchanges launched by the owner so far
  unsigned int err;                       // sticky: a peer did not arrive within the spin limit
  unsigned int pad[30];
  unsigned int flag[2][XCHG_MAXR][32];    // [parity][source rank]: one 128-byte line each
  float data[2][XCHG_MAXR][XCHG_NV];      // [parity][source rank][value]
};

struct XchgPeers {
  XchgBuf* buf[XCHG_MAXR];
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_relaxed_sys(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// payload layout (all summed over ranks):
//   0 det0 numerator   1 det0 sum(mask)   2 det1 numerator   3 det1 sum(mask)
//   4 desc num(loss)   5 desc num(pos)    6 desc num(neg)    7 desc sum(mask_valid)   8 local batch size
//   9 sem0 sum        10 sem0 count      11 sem1 sum        12 sem1 count
__global__ void __launch_bounds__(32)
loss_exchange_kernel(XchgPeers peers, int rank, int world, float* __restrict__ det0, float* __restrict__ det1,
                     float* __restrict__ desc8, float* __restrict__ sem0, float* __restrict__ sem1, float B_local,
                     float Hc, float Wc, float lambda_loss, float* __restrict__ total, unsigned long long spin_ns) {
  const int lane = threadIdx.x;
  XchgBuf* L = peers.buf[rank];
  unsigned int seq = 0;
  if (lane == 0) {
    seq = L->seq + 1u;
    L->seq = seq;
  }
  seq = __shfl_sync(0xffffffffu, seq, 0);
  const int par = (int)(seq & 1u);

  float v = 0.f;
  switch (lane) {
    case 0: v = det0 ? det0[1] : 0.f; break;
    case 1: v = det0 ? det0[2] - 1e-5f : 0.f; break;
    case 2: v = det1 ? det1[1] : 0.f; break;
    case 3: v = det1 ? det1[2] - 1e-5f : 0.f; break;
    case 4: case 5: case 6: case 7: v = desc8 ? desc8[lane] : 0.f; break;
    case 8: v = B_local; break;
    case 9: v = sem0 ? sem0[1] : 0.f; break;
    case 10: v = sem0 ? sem0[2] : 0.f; break;
    case 11: v = sem1 ? sem1[1] : 0.f; break;
    case 12: v = sem1 ? sem1[2] : 0.f; break;
    default: break;
  }
  // every lane r < world pushes the whole payload to rank r: gather the 16 values into each pushing lane
  float pay[XCHG_NV];
#pragma unroll
  for (int i = 0; i < XCHG_NV; ++i) pay[i] = __shfl_sync(0xffffffffu, v, i);
  if (lane < world) {
    XchgBuf* P = peers.buf[lane];
    float4* dst = reinterpret_cast<float4*>(P->data[par][rank]);
#pragma unroll
    for (int q = 0; q < XCHG_NV / 4; ++q) {
      float4 w = make_float4(pay[4 * q], pay[4 * q + 1], pay[4 * q + 2], pay[4 * q + 3]);
      asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + q), "f"(w.x), "f"(w.y), "f"(w.z), "f"(w.w)
                   : "memory");
    }
    __threadfence_system();
    st_release_sys(&P->flag[par][rank][0], seq);
  }
  // wait for everybody's payload of THIS exchange (local memory only)
  bool ok = true;
  if (lane < world) {
    const unsigned int* f = &L->flag[par][lane][0];
    const unsigned long long t0 = globaltimer_ns();
    while ((int)(ld_acquire_sys(f) - seq) < 0) {
      if (globaltimer_ns() - t0 > spin_ns) { ok = false; break; }
      __nanosleep(64);
    }
  }
  ok = __all_sync(0xffffffffu, ok);
  __threadfence_system();
  // lane i sums value i over the ranks in rank order
  float tot = 0.f;
  if (lane < XCHG_NV) {
    for (int r = 0; r < world; ++r) tot += ld_relaxed_sys(&L->data[par][r][lane]);
  }
  if (!ok) {
    tot = __int_as_float(0x7fc00000);  // a lost peer poisons every result (NaN) instead of hanging the stream
    if (lane == 0) L->err = seq;
  }
  float s[13];
#pragma unroll
  for (int i = 0; i < 13; ++i) s[i] = __shfl_sync(0xffffffffu, tot, i);
  if (lane == 0) {
    if (det0) { det0[1] = s[0]; det0[2] = s[1] + 1e-5f; det0[0] = s[0] / (s[1] + 1e-5f); }
    if (det1) { det1[1] = s[2]; det1[2] = s[3] + 1e-5f; det1[0] = s[2] / (s[3] + 1e-5f); }
    if (desc8) {
      // normalization = B_global * (sum_global(mask_valid) + 1) * Hc * Wc, same fp32 operation order as desc_finalize
      const float norm = s[8] * (s[7] + 1.f) * Hc * Wc;
      desc8[0] = s[4] / norm; desc8[1] = s[5] / norm; desc8[2] = s[6] / norm; desc8[3] = norm;
      desc8[4] = s[4]; desc8[5] = s[5]; desc8[6] = s[6]; desc8[7] = s[7];
    }
    if (sem0) { sem0[1] = s[9]; sem0[2] = s[10]; sem0[0] = s[9] / s[10]; }
    if (sem1) { sem1[1] = s[11]; sem1[2] = s[12]; sem1[0] = s[11] / s[12]; }
    // fused loss step: the weighted total of the GLOBAL-batch losses (same expression as desc_finalize on one GPU)
    if (total && det0 && det1 && desc8) *total = (det0[0] + det1[0]) + lambda_loss * desc8[0];
  }
}

extern "C" int ssp_xchg_max_ranks(void) { return XCHG_MAXR; }

// The one allocation this library makes: IPC export needs a cudaMalloc'ed base pointer (a sub-block of a caching
// allocator cannot be exported).  ipc_handle64_host receives the 64-byte cudaIpcMemHandle_t (HOST memory).
extern "C" int ssp_xchg_alloc(void** buf, void* ipc_handle64_host) {
  SSP_REQUIRE(buf, "ssp_xchg_alloc: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* p = nullptr;
  SSP_CUDA_CALL(cudaMalloc(&p, sizeof(XchgBuf)));
  cudaError_t e = cudaMemset(p, 0, sizeof(XchgBuf));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess && ipc_handle64_host) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle64_host), p);
  if (e != cudaSuccess) {
    cudaFree(p);
    ssp_set_error("ssp_xchg_alloc: %s", cudaGetErrorString(e));
    return (int)e;
  }
  *buf = p;
  return SSP_OK;
}

extern "C" int ssp_xchg_open(const void* ipc_handle64_host, void** peer_buf) {
  SSP_REQUIRE(ipc_handle64_host && peer_buf, "ssp_xchg_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle64_host, sizeof(h));
  SSP_CUDA_CALL(cudaIpcOpenMemHandle(peer_buf, h, cudaIpcMemLazyEnablePeerAccess));
  return SSP_OK;
}

extern "C" int ssp_xchg_close(void* peer_buf) {
  if (peer_buf) SSP_CUDA_CALL(cudaIpcCloseMemHandle(peer_buf));
  return SSP_OK;
}

extern "C" int ssp_xchg_free(void* buf) {
  if (buf) SSP_CUDA_CALL(cudaFree(buf));
  return SSP_OK;
}

// Sticky error word of a local exchange buffer (0 = every exchange so far completed); synchronises the stream.
extern "C" int ssp_xchg_status(const void* local_buf, void* stream) {
  SSP_REQUIRE(local_buf, "ssp_xchg_status: null pointer");
  unsigned int err = 0;
  SSP_CUDA_CALL(cudaMemcpyAsync(&err, &reinterpret_cast<const XchgBuf*>(local_buf)->err, sizeof(err), cudaMemcpyDeviceToHost,
                                (cudaStream_t)stream));
  SSP_CUDA_CALL(cudaStreamSynchronize((cudaStream_t)stream));
  if (err) {
    ssp_set_error("loss exchange %u timed out waiting for a peer rank", err);
    return SSP_EUNSUPPORTED;
  }
  return SSP_OK;
}

// bufs_host[world]: device pointers of every rank's exchange buffer as seen from THIS process (own buffer at [rank]).
// det0 / det1: out3 of the detector losses {loss, numerator, sum(mask)+1e-5}; desc8: out8 of ssp_desc_finalize;
// sem0 / sem1: out3 of the semantic losses {loss, sum, count}.  Any of them may be NULL.  total (optional, needs det0, det1
// and desc8): det0.loss + det1.loss + lambda_loss * desc.loss of the global batch.  All are rewritten in place
// with the global-batch values.  B_local = pairs of this rank (ranks may hold different shard sizes).
extern "C" int ssp_loss_exchange(const void* const* bufs_host, int rank, int world, float* det0, float* det1, float* desc8,
                                 float* sem0, float* sem1, int B_local, int Hc, int Wc, float lambda_loss, float* total,
                                 double timeout_s, void* stream) {
  SSP_REQUIRE(bufs_host, "ssp_loss_exchange: null pointer");
  SSP_REQUIRE(world >= 1 && world <= XCHG_MAXR && rank >= 0 && rank < world, "ssp_loss_exchange: bad rank %d / world %d (max %d)",
              rank, world, XCHG_MAXR);
  SSP_REQUIRE(!desc8 || (B_local > 0 && Hc > 0 && Wc > 0), "ssp_loss_exchange: bad sizes");
  XchgPeers peers;
  for (int r = 0; r < XCHG_MAXR; ++r) peers.buf[r] = nullptr;
  for (int r = 0; r < world; ++r) {
    SSP_REQUIRE(bufs_host[r], "ssp_loss_exchange: buffer of rank %d is null", r);
    peers.buf[r] = reinterpret_cast<XchgBuf*>(const_cast<void*>(bufs_host[r]));
  }
  if (!(timeout_s > 0.0)) timeout_s = 30.0;
  loss_exchange_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(peers, rank, world, det0, det1, desc8, sem0, sem1, (float)B_local,
                                                            (float)Hc, (float)Wc, lambda_loss, total, (unsigned long long)(timeout_s * 1e9));
  SSP_CUDA_CHECK_LAUNCH("loss_exchange_kernel");
  return SSP_OK;
}
