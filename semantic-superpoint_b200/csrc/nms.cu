// Keypoint extraction: getPtsFromHeatmap / nms_fast and box_nms on the GPU.
// Reference: utils/utils.py:581-609 (getPtsFromHeatmap), :653-712 (nms_fast), :612-650 (box_nms)
//            twins in models/model_wrap.py:129-192,266-293   -- Gabriel-SGama/Semantic-SuperPoint
//
// The reference walks the candidates in descending-confidence order and keeps a point iff no
// already-kept point lies in its suppression window.  For a strict total order this greedy result is
// unique and equals the fixed point of parallel rounds:
//   undecided p:  a kept point in window(p)                     -> suppressed
//                 no undecided point of higher priority in window(p) -> kept
// State transitions are monotone (undecided -> kept | suppressed) and each pixel has one writer, so
// rounds may read stale neighbour state without changing the result (a stale "undecided" only delays
// a decision).  Priority = (confidence desc, linear index asc) = numpy stable argsort(-conf).
// The window is a (2R+1)^2 boolean stencil in shared memory: all ones for nms_fast (Chebyshev
// radius R), the IoU > thr footprint for box_nms.  Tiles are 32x32 with an R halo; each launch runs
// NMS_LOCAL_ITERS rounds on its tile snapshot before publishing.
#include "common.cuh"

#define NT 32
#define NMS_LOCAL_ITERS 4
#define ST_NONE 0
#define ST_UNDECIDED 1
#define ST_KEPT 2

__global__ void nms_init_kernel(const float* __restrict__ heat, size_t n, float thr, int strict,
                                uint8_t* __restrict__ state) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = heat[i];
  bool c = strict ? (v > thr) : (v >= thr);
  state[i] = c ? ST_UNDECIDED : ST_NONE;
}

__global__ void __launch_bounds__(256)
nms_round_kernel(const float* __restrict__ heat, uint8_t* __restrict__ state, int H, int W, int R,
                 const uint8_t* __restrict__ stencil, unsigned int* __restrict__ remaining) {
  extern __shared__ unsigned char smem_raw[];
  int TW = NT + 2 * R;
  float* sv = reinterpret_cast<float*>(smem_raw);                 // TW*TW values
  uint8_t* ss = reinterpret_cast<uint8_t*>(sv + TW * TW);         // TW*TW states
  uint8_t* sk = ss + TW * TW;                                     // (2R+1)^2 stencil
  __shared__ int any_undecided;
  int tid = threadIdx.x;
  size_t img = (size_t)blockIdx.z * H * W;
  heat += img;
  state += img;
  int ty0 = blockIdx.y * NT, tx0 = blockIdx.x * NT;
  if (tid == 0) any_undecided = 0;
  __syncthreads();
  // interior first: skip the tile when nothing is undecided
  int found = 0;
  for (int i = tid; i < NT * NT; i += 256) {
    int y = ty0 + i / NT, x = tx0 + i % NT;
    if (y < H && x < W && state[(size_t)y * W + x] == ST_UNDECIDED) found = 1;
  }
  if (found) any_undecided = 1;
  __syncthreads();
  if (!any_undecided) return;
  int S = 2 * R + 1;
  for (int i = tid; i < S * S; i += 256) sk[i] = stencil[i];
  for (int i = tid; i < TW * TW; i += 256) {
    int y = ty0 - R + i / TW, x = tx0 - R + i % TW;
    uint8_t s = ST_NONE;
    float v = 0.f;
    if (y >= 0 && y < H && x >= 0 && x < W) {
      s = state[(size_t)y * W + x];
      if (s != ST_NONE) v = heat[(size_t)y * W + x];
    }
    ss[i] = s;
    sv[i] = v;
  }
  __syncthreads();
  int left = 0;
  for (int it = 0; it < NMS_LOCAL_ITERS; ++it) {
    uint8_t ns[4];
    left = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int i = tid + q * 256;
      int ly = i / NT, lx = i % NT;
      int c = (ly + R) * TW + (lx + R);
      uint8_t s = ss[c];
      ns[q] = s;
      if (s != ST_UNDECIDED) continue;
      float v = sv[c];
      bool kept_near = false, higher_near = false;
      for (int dy = -R; dy <= R; ++dy) {
        for (int dx = -R; dx <= R; ++dx) {
          if (!sk[(dy + R) * S + (dx + R)] || (dx == 0 && dy == 0)) continue;
          int o = c + dy * TW + dx;
          uint8_t so = ss[o];
          if (so == ST_KEPT) kept_near = true;
          else if (so == ST_UNDECIDED) {
            float vo = sv[o];
            // priority: larger value first, then smaller linear index (dy<0 or dy==0&&dx<0)
            if (vo > v || (vo == v && (dy < 0 || (dy == 0 && dx < 0)))) higher_near = true;
          }
        }
      }
      if (kept_near) ns[q] = ST_NONE;
      else if (!higher_near) ns[q] = ST_KEPT;
      else left++;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int i = tid + q * 256;
      ss[(i / NT + R) * TW + (i % NT + R)] = ns[q];
    }
    __syncthreads();
  }
  // publish the interior
  for (int i = tid; i < NT * NT; i += 256) {
    int y = ty0 + i / NT, x = tx0 + i % NT;
    if (y < H && x < W) state[(size_t)y * W + x] = ss[(i / NT + R) * TW + (i % NT + R)];
  }
  if (left) atomicAdd(remaining, (unsigned int)left);
}

// Priority as one unique 64-bit key (order-preserving float bits << 32 | ~linear index): larger key = higher priority.
__device__ __forceinline__ unsigned long long nms_key(float v, unsigned int idx) {
  unsigned int u = __float_as_uint(v);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - idx);
}

// Square-window rounds, sliding-window form (R known at compile time).  One 64-bit array carries everything a round needs:
//   key = 0                suppressed / not a candidate
//   key = all ones         kept
//   otherwise              undecided, its priority (order-preserving value bits << 32 | ~linear index)
// so "a kept point in my window" and "I am the highest undecided point of my window" are the SAME window maximum m:
// m == all ones -> suppressed, m == own key -> kept.  The (2R+1)^2 maximum is separable, and each thread produces several
// adjacent outputs of a pass from registers: S outputs need S + 2R inputs and ~(S + 2R) log2(2R+1) max operations
// (doubling: windows of 1, 2, 4, ... then one overlap step), instead of S (2R+1) shared-memory reads each.
template <int W, int N>
__device__ __forceinline__ void sliding_max(unsigned long long (&a)[N]) {
  int p = 1;
#pragma unroll
  for (int step = 0; step < 5; ++step) {
    if (2 * p <= W) {
#pragma unroll
      for (int i = 0; i < N; ++i)
        if (i + p < N) a[i] = max(a[i], a[i + p]);
      p *= 2;
    }
  }
  if (p < W) {
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (i + W - p < N) a[i] = max(a[i], a[i + W - p]);
  }
}

template <int R>
__global__ void __launch_bounds__(256)
nms_round_sliding_kernel(const float* __restrict__ heat, uint8_t* __restrict__ state, int H, int W,
                         unsigned int* __restrict__ remaining) {
  constexpr int TW = NT + 2 * R;
  constexpr unsigned long long ONES = ~0ull;
  __shared__ unsigned long long key[TW][TW + 1];
  __shared__ unsigned long long rm[TW][NT + 1];  // row maxima of the interior columns, all TW rows
  const int tid = threadIdx.x;
  const size_t img = (size_t)blockIdx.z * H * W;
  heat += img;
  state += img;
  const int ty0 = blockIdx.y * NT, tx0 = blockIdx.x * NT;
  int found = 0;
  for (int i = tid; i < NT * NT; i += 256) {
    const int y = ty0 + i / NT, x = tx0 + i % NT;
    if (y < H && x < W && state[(size_t)y * W + x] == ST_UNDECIDED) found = 1;
  }
  if (!__syncthreads_or(found)) return;  // converged tile: one read of its own state
  for (int i = tid; i < TW * TW; i += 256) {
    const int ly = i / TW, lx = i - ly * TW;
    const int y = ty0 - R + ly, x = tx0 - R + lx;
    unsigned long long k = 0ull;
    if (y >= 0 && y < H && x >= 0 && x < W) {
      const uint8_t st = state[(size_t)y * W + x];
      if (st == ST_KEPT) k = ONES;
      else if (st == ST_UNDECIDED) k = nms_key(heat[(size_t)y * W + x], (unsigned int)(y * W + x));
    }
    key[ly][lx] = k;
  }
  __syncthreads();
  constexpr int SR = 8, SC = 4;  // outputs per thread: row pass (TW rows x 4 segments), column pass (32 columns x 8 segments)
  for (int it = 0; it < NMS_LOCAL_ITERS; ++it) {
    if (tid < TW * (NT / SR)) {
      const int row = tid / (NT / SR), c0 = (tid % (NT / SR)) * SR;
      unsigned long long a[SR + 2 * R];
#pragma unroll
      for (int j = 0; j < SR + 2 * R; ++j) a[j] = key[row][c0 + j];
      sliding_max<2 * R + 1, SR + 2 * R>(a);
#pragma unroll
      for (int j = 0; j < SR; ++j) rm[row][c0 + j] = a[j];
    }
    __syncthreads();
    int changed = 0;
    {
      const int col = tid & (NT - 1), r0 = (tid / NT) * SC;
      unsigned long long a[SC + 2 * R];
#pragma unroll
      for (int j = 0; j < SC + 2 * R; ++j) a[j] = rm[r0 + j][col];
      sliding_max<2 * R + 1, SC + 2 * R>(a);
#pragma unroll
      for (int j = 0; j < SC; ++j) {
        const unsigned long long k = key[r0 + j + R][col + R];
        if (k != 0ull && k != ONES) {
          if (a[j] == ONES) { key[r0 + j + R][col + R] = 0ull; changed = 1; }
          else if (a[j] == k) { key[r0 + j + R][col + R] = ONES; changed = 1; }
        }
      }
    }
    if (!__syncthreads_or(changed)) break;  // nothing moved: further rounds on this snapshot cannot either
  }
  int left = 0;
  for (int i = tid; i < NT * NT; i += 256) {
    const int ly = i / NT, lx = i % NT;
    const int y = ty0 + ly, x = tx0 + lx;
    if (y < H && x < W) {
      const unsigned long long k = key[ly + R][lx + R];
      const uint8_t st = k == 0ull ? ST_NONE : (k == ONES ? ST_KEPT : ST_UNDECIDED);
      left += st == ST_UNDECIDED;
      state[(size_t)y * W + x] = st;
    }
  }
  if (left) atomicAdd(remaining, (unsigned int)left);
}

template <int R>
static void launch_sliding(dim3 grid, const float* heat, uint8_t* state, int H, int W, unsigned int* remaining, cudaStream_t st) {
  nms_round_sliding_kernel<R><<<grid, 256, 0, st>>>(heat, state, H, W, remaining);
}

// true when a compiled sliding-window instance exists for this radius
static bool nms_launch_sliding(int R, dim3 grid, const float* heat, uint8_t* state, int H, int W, unsigned int* remaining,
                               cudaStream_t st) {
  switch (R) {
    case 1: launch_sliding<1>(grid, heat, state, H, W, remaining, st); return true;
    case 2: launch_sliding<2>(grid, heat, state, H, W, remaining, st); return true;
    case 3: launch_sliding<3>(grid, heat, state, H, W, remaining, st); return true;
    case 4: launch_sliding<4>(grid, heat, state, H, W, remaining, st); return true;
    case 5: launch_sliding<5>(grid, heat, state, H, W, remaining, st); return true;
    case 6: launch_sliding<6>(grid, heat, state, H, W, remaining, st); return true;
    case 7: launch_sliding<7>(grid, heat, state, H, W, remaining, st); return true;
    case 8: launch_sliding<8>(grid, heat, state, H, W, remaining, st); return true;
    default: return false;
  }
}

// kept points outside the removed border -> unordered list (value, linear index)
__global__ void nms_compact_kernel(const float* __restrict__ heat, const uint8_t* __restrict__ state, int H, int W,
                                   int border, int capacity, float* __restrict__ lval, int* __restrict__ lidx,
                                   unsigned int* __restrict__ count) {
  int img = blockIdx.y;
  size_t off = (size_t)img * H * W;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  if (i < H * W) {
    int y = i / W, x = i % W;
    keep = state[off + i] == ST_KEPT && x >= border && x < W - border && y >= border && y < H - border;
  }
  unsigned int bal = __ballot_sync(0xffffffffu, keep);
  int lane = threadIdx.x & 31;
  unsigned int base = 0;
  if (lane == 0 && bal) base = atomicAdd(count + img, (unsigned int)__popc(bal));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (keep) {
    unsigned int slot = base + __popc(bal & ((1u << lane) - 1u));
    if (slot < (unsigned int)capacity) {
      lval[(size_t)img * capacity + slot] = heat[off + i];
      lidx[(size_t)img * capacity + slot] = i;
    }
  }
}

// rank-by-counting sort: output order = (confidence desc, linear index desc), i.e. the reference's
// `argsort(conf)[::-1]` with a stable sort.  pts is [3, capacity] doubles per image: x, y, conf.
__global__ void __launch_bounds__(256)
nms_rank_emit_kernel(const float* __restrict__ lval, const int* __restrict__ lidx,
                     const unsigned int* __restrict__ count, int W, int capacity, double* __restrict__ pts) {
  __shared__ float tv[256];
  __shared__ int ti[256];
  int img = blockIdx.y;
  int K = min((int)count[img], capacity);
  lval += (size_t)img * capacity;
  lidx += (size_t)img * capacity;
  pts += (size_t)img * 3 * capacity;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x * blockDim.x >= K) return;
  float v = 0.f;
  int id = 0;
  if (i < K) { v = lval[i]; id = lidx[i]; }
  int rank = 0;
  for (int base = 0; base < K; base += 256) {
    int j = base + threadIdx.x;
    __syncthreads();
    if (j < K) { tv[threadIdx.x] = lval[j]; ti[threadIdx.x] = lidx[j]; }
    __syncthreads();
    int lim = min(256, K - base);
    for (int q = 0; q < lim; ++q) {
      float vo = tv[q];
      int io = ti[q];
      rank += (vo > v || (vo == v && io > id)) ? 1 : 0;
    }
  }
  if (i < K) {
    pts[rank] = (double)(id % W);
    pts[capacity + rank] = (double)(id / W);
    pts[2 * (size_t)capacity + rank] = (double)v;
  }
}

__global__ void nms_dense_kernel(const float* __restrict__ heat, const uint8_t* __restrict__ state, size_t n,
                                 float* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = state[i] == ST_KEPT ? heat[i] : 0.f;
}

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
extern "C" size_t ssp_nms_ws_bytes(int I, int H, int W, int capacity) {
  size_t n = (size_t)I * H * W;
  size_t state = (n + 255) / 256 * 256;
  size_t ctr = 256 + (((size_t)I * 4 + 255) / 256) * 256;   // [remaining | pad] + per-image counts
  size_t lists = (size_t)I * capacity * 8;
  return state + ctr + lists + 256;
}

// workspace: state map (rounded to 256 B) | round counter (256 B) | per-image keypoint counts | candidate lists
extern "C" size_t ssp_nms_ws_counts_offset(int I, int H, int W) {
  return ((size_t)I * H * W + 255) / 256 * 256 + 256;
}

struct NmsWs {
  uint8_t* state;
  unsigned int* remaining;
  unsigned int* count;
  float* lval;
  int* lidx;
};

static NmsWs nms_carve(void* ws, int I, int H, int W, int capacity) {
  NmsWs w;
  size_t n = (size_t)I * H * W;
  char* p = (char*)ws;
  w.state = (uint8_t*)p;
  w.remaining = (unsigned int*)(p + (n + 255) / 256 * 256);
  p += ssp_nms_ws_counts_offset(I, H, W);
  w.count = (unsigned int*)p;
  p += (((size_t)I * 4 + 255) / 256) * 256;
  w.lval = (float*)p;
  p += (size_t)I * capacity * 4;
  w.lidx = (int*)p;
  return w;
}

// Runs the rounds to the fixed point.  Synchronises the stream every `batch` rounds to read the
// number of still-undecided pixels (the reference API returns host data, so a sync is inherent).
// square: the stencil is the full (2R+1)^2 window (nms_fast), so radii 1..8 run the sliding-window kernel; every other
// radius, and every box_nms footprint, runs the stencil kernel.  Both reach the greedy result for the order (confidence
// desc, linear index asc); the only difference is that the 64-bit key orders -0.0 below +0.0 where the float compare of
// the stencil kernel ties them.  That matters only when both signed zeros are candidates at once, which no caller
// produces: flattenDetection heatmaps are >= +0, and utils.nms_fast has one -0.0 among negative ranks and NaN.
static int nms_run_rounds(const float* heat, const NmsWs& w, int I, int H, int W, int R, const uint8_t* stencil,
                          bool square, cudaStream_t st) {
  dim3 grid(ssp_ceil_div(W, NT), ssp_ceil_div(H, NT), I);
  int TW = NT + 2 * R;
  size_t smem = (size_t)TW * TW * 5 + (size_t)(2 * R + 1) * (2 * R + 1);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(nms_round_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { ssp_set_error("nms: window radius %d needs %zu B shared memory: %s", R, smem, cudaGetErrorString(e)); return (int)e; }
  }
  int rounds = 0;
  unsigned int remaining = 1;
  // dense random maps converge in 7-9 launches (4 local rounds each), real heatmaps in 2-3; a converged tile leaves after one
  // read of its own state (~4 us per launch for 32 images), a host check costs a stream sync: 8 launches, then 4 at a time
  int batch = 8;
  while (remaining) {
    for (int k = 0; k < batch; ++k) {
      if (k == batch - 1) SSP_CUDA_CALL(cudaMemsetAsync(w.remaining, 0, 4, st));
      if (!(square && nms_launch_sliding(R, grid, heat, w.state, H, W, w.remaining, st)))
        nms_round_kernel<<<grid, 256, smem, st>>>(heat, w.state, H, W, R, stencil, w.remaining);
      SSP_CUDA_CHECK_LAUNCH("nms_round_kernel");
      ++rounds;
    }
    batch = 4;
    SSP_CUDA_CALL(cudaMemcpyAsync(&remaining, w.remaining, 4, cudaMemcpyDeviceToHost, st));
    SSP_CUDA_CALL(cudaStreamSynchronize(st));
    if (rounds > 4 * (H + W) * I + 64) { ssp_set_error("nms: rounds did not converge"); return SSP_EUNSUPPORTED; }
  }
  return SSP_OK;
}

// getPtsFromHeatmap for I images of HxW.  pts: [I,3,capacity] float64 (x,y,conf rows, conf-descending),
// counts_host: [I] ints on the HOST (number of points per image).  stencil: device (2R+1)^2 bytes.
extern "C" int ssp_nms_fast(const float* heat, int I, int H, int W, float conf_thresh, int R,
                            const uint8_t* stencil, int border, int capacity, double* pts, int* counts_host,
                            void* ws, size_t ws_bytes, void* stream) {
  SSP_REQUIRE(heat && stencil && pts && counts_host && ws, "ssp_nms_fast: null pointer");
  SSP_REQUIRE(I > 0 && I <= 65535 && H > 0 && W > 0 && R >= 0 && R <= 48 && border >= 0 && capacity > 0,
              "ssp_nms_fast: bad sizes I=%d H=%d W=%d R=%d border=%d capacity=%d", I, H, W, R, border, capacity);
  SSP_REQUIRE(ws_bytes >= ssp_nms_ws_bytes(I, H, W, capacity), "ssp_nms_fast: workspace too small");
  SSP_REQUIRE(((uintptr_t)ws & 255) == 0, "ssp_nms_fast: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  NmsWs w = nms_carve(ws, I, H, W, capacity);
  size_t n = (size_t)I * H * W;
  nms_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(heat, n, conf_thresh, 0, w.state);
  SSP_CUDA_CHECK_LAUNCH("nms_init_kernel");
  // the stencil of nms_fast is the full (2R+1)^2 square (all ones)
  int rc = nms_run_rounds(heat, w, I, H, W, R, stencil, true, st);
  if (rc) return rc;
  SSP_CUDA_CALL(cudaMemsetAsync(w.count, 0, (size_t)I * 4, st));
  dim3 cg(ssp_ceil_div(H * W, 256), I);
  nms_compact_kernel<<<cg, 256, 0, st>>>(heat, w.state, H, W, border, capacity, w.lval, w.lidx, w.count);
  SSP_CUDA_CHECK_LAUNCH("nms_compact_kernel");
  dim3 rg(ssp_ceil_div(capacity, 256), I);
  nms_rank_emit_kernel<<<rg, 256, 0, st>>>(w.lval, w.lidx, w.count, W, capacity, pts);
  SSP_CUDA_CHECK_LAUNCH("nms_rank_emit_kernel");
  SSP_CUDA_CALL(cudaMemcpyAsync(counts_host, w.count, (size_t)I * 4, cudaMemcpyDeviceToHost, st));
  SSP_CUDA_CALL(cudaStreamSynchronize(st));
  for (int i = 0; i < I; ++i) {
    if (counts_host[i] > capacity) {
      ssp_set_error("ssp_nms_fast: image %d has %d keypoints, capacity %d", i, counts_host[i], capacity);
      return SSP_EARG;
    }
  }
  return SSP_OK;
}

// box_nms: candidates prob > min_prob (strict), IoU-footprint stencil, dense output map.
extern "C" int ssp_box_nms(const float* prob, int I, int H, int W, float min_prob, int R, const uint8_t* stencil,
                           float* out, void* ws, size_t ws_bytes, void* stream) {
  SSP_REQUIRE(prob && stencil && out && ws, "ssp_box_nms: null pointer");
  SSP_REQUIRE(I > 0 && I <= 65535 && H > 0 && W > 0 && R >= 0 && R <= 48, "ssp_box_nms: bad sizes I=%d H=%d W=%d R=%d", I, H, W, R);
  SSP_REQUIRE(ws_bytes >= ssp_nms_ws_bytes(I, H, W, 1), "ssp_box_nms: workspace too small");
  SSP_REQUIRE(((uintptr_t)ws & 255) == 0, "ssp_box_nms: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  NmsWs w = nms_carve(ws, I, H, W, 1);
  size_t n = (size_t)I * H * W;
  nms_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(prob, n, min_prob, 1, w.state);
  SSP_CUDA_CHECK_LAUNCH("nms_init_kernel");
  int rc = nms_run_rounds(prob, w, I, H, W, R, stencil, false, st);
  if (rc) return rc;
  nms_dense_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(prob, w.state, n, out);
  SSP_CUDA_CHECK_LAUNCH("nms_dense_kernel");
  return SSP_OK;
}
