// Shared pieces of the fused per-pixel kernels: parameters, PTX wrappers (mbarrier + 1-D TMA
// bulk copies), vector access helpers and the per-pixel loss / gradient-coefficient stage.
#pragma once
#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "common.cuh"

namespace bacs {

constexpr int kConsumerWarps = 8;
constexpr int kConsumers = 32 * kConsumerWarps;
constexpr int kMaxStages = 4;

struct alignas(64) PixelParams {
  CUtensorMap tmap_in;   // logits   as a 3-D tensor (H*W, K, B), box (256, K, 1)  -- fast path only
  CUtensorMap tmap_out;  // dlogits, same geometry
  CUtensorMap tmap_z;    // seen logits as (w, h, T, B), box (w, 2, T, 1): both source rows of every head
  int use_tmap;
  bacs_pixel_args a;
  int P;                // pixels per tile
  int tiles_per_image;
  int n_tiles;
  int stages;
  int use_bulk;         // rows are 16-byte aligned -> TMA bulk copies
  float inv_n;          // 1 / (B*H*W)
  float sy, sx;         // align_corners=True scales (h-1)/(H-1), (w-1)/(W-1)
  double* partials;     // [gridDim.x, BACS_NACC]  (SCORE mode: [n_tiles, BACS_NACC])
};

// ---- PTX wrappers: mbarrier + 1-D bulk async copy (TMA) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
// 3-D tiled TMA (tensor map in kernel-parameter space): whole [K][256] boxes per instruction
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst_smem)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
          smem_u32(dst_smem)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, int c0, int c1, int c2, const void* src_smem) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
               "r"(smem_u32(src_smem)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "elect.sync _|P1, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory"); }

__device__ __forceinline__ float ex2_fast(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ---- vector access to PPT adjacent pixels of one shared-memory row -------------------
template <typename T, int PPT> struct Vec;
template <> struct Vec<float, 1> {
  __device__ static __forceinline__ void ld(const float* p, float* v) { v[0] = p[0]; }
  __device__ static __forceinline__ void st(float* p, const float* v) { p[0] = v[0]; }
};
template <> struct Vec<float, 2> {
  __device__ static __forceinline__ void ld(const float* p, float* v) {
    const float2 t = *reinterpret_cast<const float2*>(p);
    v[0] = t.x; v[1] = t.y;
  }
  __device__ static __forceinline__ void st(float* p, const float* v) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  }
};
template <> struct Vec<__nv_bfloat16, 1> {
  __device__ static __forceinline__ void ld(const __nv_bfloat16* p, float* v) { v[0] = __bfloat162float(p[0]); }
  __device__ static __forceinline__ void st(__nv_bfloat16* p, const float* v) { p[0] = __float2bfloat16_rn(v[0]); }
};
template <> struct Vec<__nv_bfloat16, 2> {
  __device__ static __forceinline__ void ld(const __nv_bfloat16* p, float* v) {
    const float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
    v[0] = t.x; v[1] = t.y;
  }
  __device__ static __forceinline__ void st(__nv_bfloat16* p, const float* v) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(v[0], v[1]);
  }
};
template <> struct Vec<__half, 1> {
  __device__ static __forceinline__ void ld(const __half* p, float* v) { v[0] = __half2float(p[0]); }
  __device__ static __forceinline__ void st(__half* p, const float* v) { p[0] = __float2half_rn(v[0]); }
};
template <> struct Vec<__half, 2> {
  __device__ static __forceinline__ void ld(const __half* p, float* v) {
    const float2 t = __half22float2(*reinterpret_cast<const __half2*>(p));
    v[0] = t.x; v[1] = t.y;
  }
  __device__ static __forceinline__ void st(__half* p, const float* v) {
    *reinterpret_cast<__half2*>(p) = __floats2half2_rn(v[0], v[1]);
  }
};

__device__ __forceinline__ float pow_gamma(float base, float gamma) {
  if (gamma == 2.f) return base * base;
  if (gamma == 1.f) return base;
  if (gamma == 0.f) return 1.f;
  return powf(base, gamma);
}

constexpr float kLog2e = 1.4426950408889634f;

// Per-pixel result of the loss stage: gradient of pixel = e_k * cg[group(k)] - [k==0] d0 - [k==y] dy
// with groups 0: k == 0, 1: 1 <= k < old_cl, 2: k >= old_cl.
struct PixCoef {
  float cg0, cg1, cg2, d0, dy;
};

// Last lane of the run of consecutive lanes that holds this lane's `key`.  A segmented shfl_down tree reduction may
// add lane + o's partial sum only when lane + o <= this lane: a key can come back after a different one (a warp's
// pixels wrapping into the next image row meet the same low-res cell again), and that later run is flushed by its
// own first lane.
__device__ __forceinline__ int run_end_lane(int key, int lane) {
  const int next = __shfl_down_sync(0xffffffffu, key, 1);
  const unsigned ends = __ballot_sync(0xffffffffu, lane == 31 || next != key);
  return __ffs(ends & (0xffffffffu << lane)) - 1;
}

// Binary focal loss of one seen-head logit Z with target t (smp FocalLoss(mode="binary"), base_loss.py:255-272):
//   bce = softplus(Z) - t Z,  pt = exp(-bce) = sigmoid(+-Z),  term = (1-pt)^g * bce [* alpha weight]; dterm = d term / dZ
__device__ __forceinline__ void focal_term(const bacs_pixel_args& a, float Z, float t, float& term, float& dterm) {
  const float e = __expf(-fabsf(Z));
  const float inv = __fdividef(1.f, 1.f + e);
  const float hi = inv, lo = e * inv;                        // sigmoid(|Z|), sigmoid(-|Z|)
  const float sig = Z >= 0.f ? hi : lo;                      // sigmoid(Z)
  const float nsig = Z >= 0.f ? lo : hi;                     // 1 - sigmoid(Z) without cancellation
  const float pt = (t != 0.f) ? sig : nsig;
  const float om = (t != 0.f) ? nsig : sig;                  // 1 - pt
  const float dbce = (t != 0.f) ? -nsig : sig;               // sigmoid(Z) - t
  const float bce = fmaxf(Z, 0.f) - Z * t + __logf(1.f + e);
  if (a.focal_gamma == 2.f) {
    term = om * om * bce;
    dterm = dbce * (om * om + 2.f * om * pt * bce);
  } else if (a.focal_gamma == 0.f) {
    term = bce;
    dterm = dbce;
  } else {
    const float pg = powf(om, a.focal_gamma);
    term = pg * bce;
    dterm = dbce * (pg + a.focal_gamma * powf(om, a.focal_gamma - 1.f) * pt * bce);
  }
  if (a.focal_alpha >= 0.f) {
    const float aw = a.focal_alpha * t + (1.f - a.focal_alpha) * (1.f - t);
    term *= aw;
    dterm *= aw;
  }
}

// Everything that depends on the softmax statistics of ONE pixel (not on the channel loop).
__device__ __forceinline__ void pixel_terms(const bacs_pixel_args& a, float inv_n, float s_norm, int old_cl, int y,
                                            bool is_ign, float mx, float S, float S_old, float S_fg_in, float e0, float x0,
                                            float xy,
                                            float seen, bool have_seen, float zfoc, float* acc, PixCoef& pc,
                                            float& gfoc, uint8_t& dmask) {
  pc.cg0 = pc.cg1 = pc.cg2 = pc.d0 = pc.dy = 0.f;
  gfoc = 0.f;
  dmask = 0;
  const float logS = __logf(S);
  const float lse = mx + logS;
  const float inv_S = __fdividef(1.f, S);
  const bool valid = y >= 0;
  if (!is_ign) acc[BACS_ACC_KEPT] += 1.f;
  if (valid) acc[BACS_ACC_VALID] += 1.f;
  if (valid && y == 0) acc[BACS_ACC_BG] += 1.f;
  const float gs_bacs = inv_n * a.grad_scale;

  if (a.mode == BACS_PIX_WEIGHTED_CE) {
    if (valid) {
      // S_fg = sum over the foreground channels, accumulated WITHOUT channel 0 by the caller: S - e0 cancels
      // catastrophically when the background logit dominates (confident networks)
      const float S_fg = fmaxf(S_fg_in, 1e-37f);
      const float u = a.ukd ? 1.f : 0.f;
      const float inv_old = __fdividef(1.f, S_old);
      const float inv_fg = __fdividef(1.f, S_fg);
      const float l_old = u * (logS - __logf(S_old));
      float l1, l2;
      if (y == 0) {
        float s = seen;
        if (s > a.threshold) s = 1.f;
        const float mod = pow_gamma(1.f - s, a.gamma);
        l1 = mod * (lse - x0);
        l2 = l_old;
        pc.cg0 = mod * inv_S + u * (inv_S - inv_old);
        pc.cg1 = pc.cg0;
        pc.cg2 = mod * inv_S + u * inv_S;
        pc.d0 = mod;
      } else if (y < old_cl) {
        l1 = logS - __logf(S_fg);
        l2 = l_old;
        pc.cg0 = inv_S + u * (inv_S - inv_old);
        pc.cg1 = inv_S - inv_fg + u * (inv_S - inv_old);
        pc.cg2 = inv_S - inv_fg + u * inv_S;
      } else {
        l1 = logS - __logf(S_fg);
        l2 = lse - xy;
        pc.cg0 = 2.f * inv_S;
        pc.cg1 = 2.f * inv_S - inv_fg;
        pc.cg2 = pc.cg1;
        pc.dy = 1.f;
      }
      acc[BACS_ACC_LOSS] += l1 + l2;
      pc.cg0 *= gs_bacs; pc.cg1 *= gs_bacs; pc.cg2 *= gs_bacs; pc.d0 *= gs_bacs; pc.dy *= gs_bacs;
    }
  } else if (a.mode == BACS_PIX_CE || a.mode == BACS_PIX_SCORE) {
    if (valid) {
      const float wgt = a.class_w ? __ldg(a.class_w + y) : 1.f;
      acc[BACS_ACC_LOSS] += wgt * (lse - xy);
      acc[BACS_ACC_WSUM] += wgt;
      if (a.dlogits) {
        const float g = wgt * s_norm * a.grad_scale;
        pc.cg0 = pc.cg1 = pc.cg2 = g * inv_S;
        pc.dy = g;
      }
    }
  } else {  // BACS_PIX_UNBIASED_CE
    if (valid) {
      const float g = a.dlogits ? s_norm * a.grad_scale : 0.f;
      if (y < old_cl) {
        acc[BACS_ACC_LOSS] += logS - __logf(S_old);
        pc.cg0 = pc.cg1 = g * (inv_S - __fdividef(1.f, S_old));
        pc.cg2 = g * inv_S;
      } else {
        acc[BACS_ACC_LOSS] += lse - xy;
        pc.cg0 = pc.cg1 = pc.cg2 = g * inv_S;
        pc.dy = g;
      }
      acc[BACS_ACC_WSUM] += 1.f;
    }
  }

  // teacher-distill pixel mask: background label and confidently "seen"
  if (a.distill_mask) {
    const bool m = valid && y == 0 && (!have_seen || seen > a.lkd_threshold);
    dmask = m ? 1 : 0;
    if (m) acc[BACS_ACC_DISTILL_PIX] += 1.f;
  }

  // seen-detector focal loss of head `focal_head` (binary, target = foreground)
  if (a.gz && !is_ign) {
    float term, dterm;
    focal_term(a, zfoc, (valid && y == 0) ? 0.f : 1.f, term, dterm);
    acc[BACS_ACC_FOCAL] += term;
    gfoc = dterm;
  }
}

// The "-dy at the label's own channel" part of pixel_terms() depends on the label channel alone (same expressions,
// same rounding): kernels that reduce gradients per channel apply it once per (channel, pixel set).
__device__ __forceinline__ float label_dy(const bacs_pixel_args& a, float inv_n, float s_norm, int old_cl, int c) {
  if (a.mode == BACS_PIX_WEIGHTED_CE) return c >= old_cl ? inv_n * a.grad_scale : 0.f;
  if (a.mode == BACS_PIX_CE || a.mode == BACS_PIX_SCORE)
    return a.dlogits ? (a.class_w ? __ldg(a.class_w + c) : 1.f) * s_norm * a.grad_scale : 0.f;
  return (a.dlogits && c >= old_cl) ? s_norm * a.grad_scale : 0.f;
}

struct PixelPlan {
  int ppt, P, kreg, stages, grid, rowtile, coop;
  size_t smem;
};

// Launches a pixel kernel with `smem` bytes of dynamic shared memory, opted in when above the 48 KB default; through
// launch_pdl() when `pdl`.  `fn` (the entry point) starts the error message.
template <typename... KArgs, typename... Args>
static inline int launch_pixel_kernel(const char* fn, bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block,
                                      size_t smem, cudaStream_t s, Args... args) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("%s: cannot opt in to %zu bytes of shared memory: %s", fn, smem, cudaGetErrorString(e));
      return BACS_ERR_CUDA;
    }
  }
  if (pdl) launch_pdl(kern, grid, block, smem, s, args...);
  else kern<<<grid, block, smem, s>>>(static_cast<KArgs>(args)...);
  return BACS_OK;
}

// launchers of the register-resident fast path, one translation unit per storage type
int launch_pixel_fast_f32(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);
int launch_pixel_fast_bf16(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);
int launch_pixel_fast_f16(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);
// launchers of the training-step specialisation (pixel_wce.cuh)
int launch_pixel_wce_f32(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);
int launch_pixel_wce_bf16(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);
int launch_pixel_wce_f16(const PixelParams& p, const PixelPlan& plan, cudaStream_t s);

}  // namespace bacs
