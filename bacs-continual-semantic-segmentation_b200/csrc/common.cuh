// Shared device/host helpers for libbacs_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "bacs_b200.h"

#define BACS_VERSION 100

namespace bacs {

void set_error(const char* fmt, ...);

#define BACS_REQUIRE(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      bacs::set_error(__VA_ARGS__);  \
      return BACS_ERR_INVALID;       \
    }                                \
  } while (0)

extern unsigned long long g_launch_count;

#define BACS_CHECK_LAUNCH(name)                                               \
  do {                                                                        \
    ++bacs::g_launch_count;                                                   \
    cudaError_t e__ = cudaGetLastError();                                     \
    if (e__ != cudaSuccess) {                                                 \
      bacs::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return BACS_ERR_CUDA;                                                   \
    }                                                                         \
  } while (0)

int sm_count();

constexpr int kMaxTasks = BACS_MAX_TASKS;

// ---- programmatic dependent launch ---------------------------------------------------
// The kernels of a training step run back to back on one stream.  Launched through launch_pdl() a kernel may become
// resident while its predecessor drains: everything before pdl_wait() (shared-memory tables, barrier and tensor-memory
// set-up, index arithmetic) overlaps the predecessor's tail; pdl_wait() returns once the predecessor has completed and
// flushed, so every access to memory another kernel of the stream produces or still reads comes after it.  EVERY
// thread of a kernel launched this way calls pdl_wait() exactly once before its first such access -- a kernel that
// completed without waiting would let its own successor overtake the predecessor.  pdl_trigger() (optional) lets the
// successor start becoming resident before this grid has exited.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                     Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- storage dtype <-> float ---------------------------------------------------------
template <typename T> struct DT;
template <> struct DT<float> {
  static constexpr int id = BACS_F32;
  __device__ static __forceinline__ float to_f(float v) { return v; }
  __device__ static __forceinline__ float from_f(float v) { return v; }
};
template <> struct DT<__nv_bfloat16> {
  static constexpr int id = BACS_BF16;
  __device__ static __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct DT<__half> {
  static constexpr int id = BACS_F16;
  __device__ static __forceinline__ float to_f(__half v) { return __half2float(v); }
  __device__ static __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

static inline size_t dtype_size(int dtype) { return dtype == BACS_F32 ? 4 : 2; }

#define BACS_DISPATCH_DTYPE(dtype, T, ...)                    \
  switch (dtype) {                                            \
    case BACS_F32: { using T = float; __VA_ARGS__; } break;   \
    case BACS_BF16: { using T = __nv_bfloat16; __VA_ARGS__; } break; \
    case BACS_F16: { using T = __half; __VA_ARGS__; } break;  \
    default: bacs::set_error("unknown dtype %d", dtype); return BACS_ERR_INVALID; \
  }

// ---- warp / block reductions ---------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the block; result valid in thread 0.  `scratch` holds >= 32 T's.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? scratch[threadIdx.x] : T(0);
  if (wid == 0) r = warp_sum(r);
  return r;
}


// ---- packed fp32 pairs (sm_100 FFMA2 / FMUL2 / FADD2: two fp32 results per issued instruction) ----
// ptxas folds f2b() broadcasts and half swaps into operand modifiers (.F32, .LO_HI), so pairs built
// from one scalar cost no extra register or move.
struct F2 {
  unsigned long long v;
};
__device__ __forceinline__ F2 f2(float lo, float hi) {
  F2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ F2 f2b(float x) { return f2(x, x); }
__device__ __forceinline__ float f2lo(F2 a) {
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v));
  return lo;
}
__device__ __forceinline__ float f2hi(F2 a) {
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v));
  return hi;
}
__device__ __forceinline__ F2 fma2(F2 a, F2 b, F2 c) {
  F2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
  return r;
}
__device__ __forceinline__ F2 mul2(F2 a, F2 b) {
  F2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}
__device__ __forceinline__ F2 add2(F2 a, F2 b) {
  F2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}
__device__ __forceinline__ F2 sub2(F2 a, F2 b) {
  F2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
  return r;
}

// fast sigmoid (ex2.approx + rcp.approx, ~2 ulp): used on the bulk feature data
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
// the same two approximations issued directly (no range fix-ups: ex2.approx.ftz saturates to 0 / +inf, and
// rcp.approx.ftz(+inf) = 0): FMUL, MUFU.EX2, FADD, MUFU.RCP
__device__ __forceinline__ float sigmoid_mufu(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}
// accurate sigmoid (used where a threshold decision depends on it)
__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// Source index / weight of torch's bilinear kernels (fp32 arithmetic, matching
// area_pixel_compute_source_index in ATen/native/UpSample.h).
struct Lerp {
  int i0, i1;
  float w1;  // weight of i1; weight of i0 is 1 - w1
};
// Explicitly rounded (no FMA contraction) so the indices match an op-by-op evaluation.
__device__ __forceinline__ Lerp lerp_align_corners(int dst, int in_size, float scale) {
  // scale = (in-1)/(out-1)
  const float src = __fmul_rn(scale, (float)dst);
  Lerp l;
  l.i0 = min((int)src, in_size - 1);
  l.i1 = l.i0 + (l.i0 < in_size - 1 ? 1 : 0);
  l.w1 = __fsub_rn(src, (float)l.i0);
  return l;
}
__device__ __forceinline__ Lerp lerp_half_pixel(int dst, int in_size, float scale) {
  // scale = in/out ; src = scale*(dst+0.5)-0.5 clamped at 0
  float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  src = src < 0.f ? 0.f : src;
  Lerp l;
  l.i0 = min((int)src, in_size - 1);
  l.i1 = l.i0 + (l.i0 < in_size - 1 ? 1 : 0);
  l.w1 = __fsub_rn(src, (float)l.i0);
  return l;
}
static inline float ac_scale(int in_size, int out_size) {
  return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.f;
}
static inline float hp_scale(int in_size, int out_size) { return (float)in_size / (float)out_size; }

}  // namespace bacs
