// Pixel x class-prototype squared distance on the 5th-generation tensor cores (north_star: "tensor cores (bf16 UMMA) only
// for the pixel-by-prototype distance when K*C is large enough (ADE20K's 150 classes)"; SURVEY 8f-4).
//
//   dist2[b, k, p] = |f_bp|^2 + |c_k|^2 - 2 <f_bp, c_k>      f = features [B, D, h*w] (NCHW), c = class prototypes [Kc, D]
//
// The reference arithmetic has no such product (its per-task heads are a weighted L1 of sigmoids, networks/
// bg_detector.py:17-40; SDR's per-class terms, loss/sdr.py:120-200, touch each pixel's own class only), so this is
// the OPTIONAL per-class prototype family entry, not part of the BACS step.
//
// One hand-written kernel (tcgen05 / TMEM, no library GEMM):
//   * a persistent CTA keeps ALL prototypes in shared memory as the B operand (bf16, K-major canonical no-swizzle
//     layout: 8 x 16-byte core matrices, k-blocks Np*16 bytes apart) and their squared norms next to it;
//   * a tile is 128 pixels of one image = the 128 TMEM lanes.  NCHW features are pixel-major: warp 17 streams
//     [32 channels x 128 pixels] boxes through a shared-memory ring with TMA (pixels / channels past the end arrive as
//     zeros); a builder thread (= one pixel = one lane) reads its 32 channels of a box (conflict-free 2-byte reads),
//     packs bf16 pairs and writes them into tensor memory as the A operand (tcgen05.st, 16 columns per chunk; the four
//     builder warpgroups take chunks in turn) -- no transpose and no M-major descriptor -- and adds up |f|^2 on the way;
//   * warp 16 issues tcgen05.mma.kind::f16 (A from TMEM, B by descriptor, fp32 accumulator [128 x Np] in TMEM) chunk by
//     chunk as the builders deliver them;
//   * epilogue in the same kernel: the builders read the accumulator back (tcgen05.ld), add the norms, clamp at zero,
//     write dist2 [B, Kc, h, w] with coalesced rows and keep the arg-min (ties -> lowest class).
#include <cuda.h>

#include <algorithm>

#include "common.cuh"

namespace bacs {
namespace cd {

constexpr int kParts = 4;                            // builder warpgroups: each takes every 4th chunk and a quarter of the classes
constexpr int kBuilderWarps = 4 * kParts;
constexpr int kBuilders = 32 * kBuilderWarps;
constexpr int kThreads = 32 * (kBuilderWarps + 2);   // + MMA warp + TMA warp
constexpr int kTileM = 128;
constexpr int kChunkK = 32;             // channels per chunk: 16 TMEM columns, 2 MMAs of K = 16
constexpr int kMaxChunks = 16;          // D <= 512: the A tile takes at most 256 columns
constexpr int kColA = 256;              // accumulator in columns [0, Np), A tile in [256, 256 + Dp / 2)
constexpr int kStageBytes = kChunkK * kTileM * 2;   // one TMA box
constexpr int kMaxStages = 8;

struct Params {
  const __nv_bfloat16* feat;
  const __nv_bfloat16* protos;
  float* dist2;
  int64_t* nearest;
  int B, D, Dp, hw, Kc, Np, tiles_per_image, n_tiles, stages;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t c) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(c));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(
          smem_u32(b)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint64_t* b) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(b)) : "memory");
}
// D[tmem, 128 x N fp32] (+)= A[tmem, 128 lanes x 8 columns = 16 bf16] * B[smem descriptor, N x 16]
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t desc_lo, uint32_t desc_hi, uint32_t idesc,
                                             uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\n.reg .b64 d;\nmov.b64 d, {%2, %3};\nsetp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], d, %4, p;\n}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(desc_lo), "r"(desc_hi), "r"(idesc), "r"(acc)
      : "memory");
}
// K-major, no swizzle (layouts established with tools/ubench/umma_probe.cu): element (n, k) of a 16-bit operand at
// (n/8)*sbo + (n%8)*16 + (k/8)*lbo + (k%8)*2 bytes
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
__host__ __device__ constexpr uint32_t make_idesc_bf16(int N) {  // bf16 x bf16 -> fp32, M = 128, both operands K-major
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
}
#define CD_FENCE_BEFORE() asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory")
#define CD_FENCE_AFTER() asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory")

__device__ __forceinline__ void tmem_st16(uint32_t a, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(a),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t a, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(a)
               : "memory");
}

// shared memory: ring of TMA boxes | B operand [Dp/8 k-blocks][Np + 1 rows][16 bytes] | cc[Np] | xx[2][128] | best[2][128] |
// arg[2][128] | barriers   (one spare 16-byte slot per k-block: the 32 lanes that copy one prototype row then hit
// different banks)
__host__ __device__ inline size_t b_bytes(int Np, int Dp) { return (size_t)(Np + 1) * 16 * (Dp >> 3); }
__host__ __device__ inline size_t smem_bytes(int Np, int Dp, int stages) {
  return (size_t)stages * kStageBytes + b_bytes(Np, Dp) + (size_t)Np * 4 + 3 * kParts * kTileM * 4 +
         (kMaxChunks + 2 + 2 * kMaxStages) * 8 + 16;
}

__global__ void __launch_bounds__(kThreads, 1) class_distance_kernel(const __grid_constant__ CUtensorMap map_feat, const Params P) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint32_t s_tmem_base;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int Np = P.Np, Dp = P.Dp, KB = Dp >> 3, nchunks = (Dp + kChunkK - 1) / kChunkK;
  const uint32_t lbo = (uint32_t)(Np + 1) * 16u;
  const int S = P.stages;
  unsigned char* s_ring = smem;
  unsigned char* s_b = smem + (size_t)S * kStageBytes;
  float* s_cc = reinterpret_cast<float*>(s_b + b_bytes(Np, Dp));
  float* s_xx = s_cc + Np;                        // [kParts][128]
  float* s_best = s_xx + kParts * kTileM;         // [kParts][128]
  int* s_arg = reinterpret_cast<int*>(s_best + kParts * kTileM);
  uint64_t* bars = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_arg + kParts * kTileM) + 7) & ~(uintptr_t)7);
  uint64_t* bar_chunk = bars;                     // [kMaxChunks]: a chunk of the A tile is in tensor memory (128 arrivals)
  uint64_t* bar_dfull = bars + kMaxChunks;        // the accumulator is complete (commit)
  uint64_t* bar_dfree = bars + kMaxChunks + 1;    // every builder has read the accumulator
  uint64_t* bar_full = bars + kMaxChunks + 2;     // [S]: a TMA box has landed (expect-tx)
  uint64_t* bar_empty = bar_full + kMaxStages;    // [S]: the warpgroup that owns the stage has read it (128 arrivals)

  if (tid == 0) {
    for (int c = 0; c < kMaxChunks; ++c) mbar_init(&bar_chunk[c], 128);
    mbar_init(bar_dfull, 1);
    mbar_init(bar_dfree, 32 * kBuilderWarps);
    for (int k = 0; k < kMaxStages; ++k) {
      mbar_init(&bar_full[k], 1);
      mbar_init(&bar_empty[k], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kBuilderWarps) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // ---- the prototypes: B operand in the canonical layout (rows >= Kc and channels >= D are zero), squared norms ----
  CD_FENCE_BEFORE();
  __syncthreads();   // barriers are initialised, tensor memory is allocated
  CD_FENCE_AFTER();
  const uint32_t tmem = s_tmem_base;
  constexpr int kWork = 32 * (kBuilderWarps + 1);   // threads that fill the prototypes: everyone but the TMA warp
  if (warp == kBuilderWarps + 1) {
    // =================================================== warp 17: feature boxes through the ring, tile after tile
    // (it runs ahead of the prototype fill: the first boxes are in flight while the B operand is being written)
    if (elect_one()) {
    uint32_t g = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
      const int b = tile / P.tiles_per_image, m0 = (tile - b * P.tiles_per_image) * kTileM;
      for (int c = 0; c < nchunks; ++c, ++g) {
        const uint32_t st = g % (uint32_t)S, use = g / (uint32_t)S;
        if (use > 0) mbar_wait(&bar_empty[st], (use - 1) & 1);
        mbar_expect_tx(&bar_full[st], kStageBytes);
        tma_load_3d(s_ring + (size_t)st * kStageBytes, &map_feat, m0, c * kChunkK, b, &bar_full[st]);
      }
    }
    }
  } else {
  // asynchronous 16-byte copies (no registers, all in flight): consecutive threads take consecutive 16-byte pieces
  // of a prototype row (coalesced in global memory); the padded k-block stride spreads them over the banks
  for (int idx = tid; idx < Np * KB; idx += kWork) {
    const int n = idx / KB, kb = idx - n * KB;
    const bool ok = n < P.Kc && kb * 8 < P.D;
    const __nv_bfloat16* src = P.protos + (ok ? (size_t)n * P.D + kb * 8 : 0);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(s_b + (size_t)kb * lbo + n * 16)), "l"(src),
                 "r"(ok ? 16 : 0)
                 : "memory");
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  asm volatile("bar.sync 2, %0;" ::"n"(kWork) : "memory");
  for (int n = tid; n < Np; n += kWork) {
    float s = 0.f;
    for (int kb = 0; kb < KB; ++kb) {
      const uint4 v = *reinterpret_cast<const uint4*>(s_b + (size_t)kb * lbo + n * 16);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = __uint_as_float(w[i] << 16), b = __uint_as_float(w[i] & 0xffff0000u);
        s = fmaf(a, a, s);
        s = fmaf(b, b, s);
      }
    }
    s_cc[n] = s;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the tensor core reads what the threads wrote
  asm volatile("bar.sync 2, %0;" ::"n"(kWork) : "memory");

  if (warp < kBuilderWarps) {
    // =================================================== builders: A tile -> tensor memory, epilogue
    const int q = warp & 3, hf = warp >> 2;              // lane quarter (TMEM lanes 32q .. 32q+31), builder warpgroup
    const int ml = q * 32 + lane;                        // pixel of the tile = TMEM lane
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    const int Nh = Np / kParts;                          // accumulator columns this warpgroup turns into distances
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
      const int b = tile / P.tiles_per_image, m0 = (tile - b * P.tiles_per_image) * kTileM;
      const int m = m0 + ml;
      const bool live = m < P.hw;
      float xx = 0.f;
      // the A columns were last read by the MMAs of the previous tile: they are complete (this thread waited for the
      // accumulator of that tile before its epilogue).  Boxes are numbered over the CTA's whole run; warpgroup p takes
      // the boxes with number % 4 == p, so (the ring depth is a multiple of 4) a stage always belongs to one warpgroup
      // and each of its barriers is observed phase by phase.
      for (int c = 0; c < nchunks; ++c) {
        const uint32_t g = it * (uint32_t)nchunks + (uint32_t)c;
        if ((int)(g % (uint32_t)kParts) != hf) continue;
        const uint32_t st = g % (uint32_t)S;
        mbar_wait(&bar_full[st], (g / (uint32_t)S) & 1);
        const unsigned short* box = reinterpret_cast<const unsigned short*>(s_ring + (size_t)st * kStageBytes) + ml;
        uint32_t r[kChunkK];
#pragma unroll
        for (int j = 0; j < kChunkK; ++j) r[j] = box[j * kTileM];
        uint32_t pk[kChunkK / 2];
#pragma unroll
        for (int j = 0; j < kChunkK / 2; ++j) {
          const float a = __uint_as_float(r[2 * j] << 16), bq = __uint_as_float(r[2 * j + 1] << 16);
          xx = fmaf(a, a, xx);
          xx = fmaf(bq, bq, xx);
          pk[j] = r[2 * j] | (r[2 * j + 1] << 16);       // k even in the low half, k odd in the high half
        }
        mbar_arrive(&bar_empty[st]);                       // the box is in registers
        tmem_st16(tlane + kColA + c * (kChunkK / 2), pk);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        CD_FENCE_BEFORE();
        mbar_arrive(&bar_chunk[c]);
      }
      s_xx[hf * kTileM + ml] = xx;
      asm volatile("bar.sync 1, %0;" ::"n"(kBuilders) : "memory");
      // warpgroup (it * nchunks + r) % 4 holds the chunks c = r, r + 4, ... of this tile: adding the partials in
      // residue order r = 0..3 gives every pixel the same association wherever its tile falls in the CTA's run, so
      // the distances do not depend on the batch split or the SM count
      xx = 0.f;
#pragma unroll
      for (int r = 0; r < kParts; ++r) xx += s_xx[((it * (uint32_t)nchunks + r) & (kParts - 1)) * kTileM + ml];
      // ---- epilogue: distances of classes [hf*Nh, hf*Nh + Nh) for this pixel ----
      mbar_wait(bar_dfull, it & 1);
      CD_FENCE_AFTER();
      float best = INFINITY;
      int arg = 0x7fffffff;
      float* out = P.dist2 + (size_t)b * P.Kc * P.hw + m;
      for (int n0 = hf * Nh; n0 < (hf + 1) * Nh; n0 += 8) {
        uint32_t d[8];
        tmem_ld8(tlane + n0, d);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int n = n0 + j;
          if (n < P.Kc) {
            const float v = fmaxf(fmaf(-2.f, __uint_as_float(d[j]), xx + s_cc[n]), 0.f);
            if (live) out[(size_t)n * P.hw] = v;
            if (v < best) {
              best = v;
              arg = n;
            }
          }
        }
      }
      CD_FENCE_BEFORE();
      mbar_arrive(bar_dfree);
      if (P.nearest) {
        s_best[hf * kTileM + ml] = best;
        s_arg[hf * kTileM + ml] = arg;
        asm volatile("bar.sync 1, %0;" ::"n"(kBuilders) : "memory");
        if (hf == 0 && live) {
#pragma unroll
          for (int pt = 1; pt < kParts; ++pt) {              // equal distances: the lower class (earlier part) wins
            const float v1 = s_best[pt * kTileM + ml];
            if (v1 < best) {
              best = v1;
              arg = s_arg[pt * kTileM + ml];
            }
          }
          P.nearest[(size_t)b * P.hw + m] = arg;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kBuilders) : "memory");   // s_xx / s_best are free for the next tile
    }
  } else if (warp == kBuilderWarps) {
    // =================================================== warp 16: MMA issue
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(Np);
    const uint64_t d0 = make_desc(smem_u32(s_b), lbo, 128);
    const uint32_t d_lo = (uint32_t)d0, d_hi = (uint32_t)(d0 >> 32);
    const uint32_t kstep = (2u * lbo) >> 4;               // two k-blocks (16 channels) per MMA, in 16-byte units
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
      if (it > 0) mbar_wait(bar_dfree, (it - 1) & 1);      // the accumulator of the previous tile has been read
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(&bar_chunk[c], it & 1);
        CD_FENCE_AFTER();
        if (leader) {
          const int steps = min(kChunkK, Dp - c * kChunkK) >> 4;
          for (int s = 0; s < steps; ++s) {
            const uint32_t ks = (uint32_t)(c * (kChunkK / 16) + s);
            umma_bf16_ts(tmem, tmem + kColA + ks * 8, d_lo + ks * kstep, d_hi, idesc, (c | s) != 0);
          }
          if (c == nchunks - 1) umma_commit(bar_dfull);
        }
        __syncwarp();
      }
    }
  }
  }
  CD_FENCE_BEFORE();
  __syncthreads();
  if (warp == kBuilderWarps) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ---- per-class segmented sums (the segmented reduction of prototypes.cu with G = K classes instead of <= 32 tasks) ----
// One warp per (image, channel) row; a lane keeps a private column of the warp's [K][32] shared-memory table, so the
// update of a pixel touches only the lane's own bank (no atomics, no conflicts), then the K rows are summed over the
// lanes.  partial[b][c][k] fp32; a second launch adds the images in fp64.
constexpr int kSumWarps = 8;
template <typename T>
__global__ void __launch_bounds__(32 * kSumWarps) class_sums_kernel(const T* __restrict__ feat, int D, int hw,
                                                                    const int64_t* __restrict__ labels, int K, int warps,
                                                                    int vec, float* __restrict__ partial) {
  extern __shared__ __align__(16) float s_tab[];   // [warps][K][32]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y, c = blockIdx.x * warps + wid;
  if (wid >= warps || c >= D) return;
  float* acc = s_tab + (size_t)wid * K * 32;
  for (int i = lane; i < K * 8; i += 32) reinterpret_cast<float4*>(acc)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  const T* row = feat + ((int64_t)b * D + c) * hw;
  const int64_t* lab = labels + (int64_t)b * hw;
  if (vec) {  // hw % 8 == 0, 16-byte aligned rows: a lane takes 8 consecutive pixels per step (one 16-byte feature load)
    static_assert(sizeof(T) == 2 || sizeof(T) == 4, "feature type");
    const int items = hw >> 3;
    for (int it0 = 0; it0 < items; it0 += 64) {
      longlong2 l2[2][4];
      uint4 raw[2][sizeof(T) / 2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int it = it0 + u * 32 + lane;
        if (it < items) {
#pragma unroll
          for (int k = 0; k < 4; ++k) l2[u][k] = __ldg(reinterpret_cast<const longlong2*>(lab + it * 8) + k);
#pragma unroll
          for (int k = 0; k < (int)(sizeof(T) / 2); ++k) raw[u][k] = __ldg(reinterpret_cast<const uint4*>(row + it * 8) + k);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (it0 + u * 32 + lane < items) {
          const T* e8 = reinterpret_cast<const T*>(&raw[u][0]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const long long l = (e & 1) ? l2[u][e >> 1].y : l2[u][e >> 1].x;
            if (l >= 0 && l < K) acc[(int)l * 32 + lane] += DT<T>::to_f(e8[e]);
          }
        }
      }
    }
  }
  constexpr int U = 8;   // independent loads in flight per lane
  for (int q0 = vec ? hw : 0; q0 < hw; q0 += 32 * U) {
    long long l[U];
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u * 32 + lane;
      l[u] = q < hw ? __ldg(lab + q) : -1;
      v[u] = q < hw ? DT<T>::to_f(row[q]) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (l[u] >= 0 && l[u] < K) acc[(int)l[u] * 32 + lane] += v[u];
  }
  __syncwarp();
  // The K column sums of the warp as a reduce-scatter over groups of 16 classes: after the exchange with lane ^ 16 a
  // lane keeps 8 classes, then 4, 2, 1 -- 16 shuffles per group instead of 5 per class (K = 151: 1 660 -> 770
  // instructions per row), with the association of warp_sum() ((l, l^16), then ^8, ^4, ^2, ^1): bit-identical sums.
  float* out = partial + ((int64_t)b * D + c) * K;
  for (int k0 = 0; k0 < K; k0 += 16) {
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = k0 + i < K ? acc[(k0 + i) * 32 + lane] : 0.f;
    float k8[8], k4[4], k2[2];
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) k8[i] = (b4 ? v[i + 8] : v[i]) + __shfl_xor_sync(0xffffffffu, b4 ? v[i] : v[i + 8], 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) k4[i] = (b3 ? k8[i + 4] : k8[i]) + __shfl_xor_sync(0xffffffffu, b3 ? k8[i] : k8[i + 4], 8);
#pragma unroll
    for (int i = 0; i < 2; ++i) k2[i] = (b2 ? k4[i + 2] : k4[i]) + __shfl_xor_sync(0xffffffffu, b2 ? k4[i] : k4[i + 2], 4);
    float k1 = (b1 ? k2[1] : k2[0]) + __shfl_xor_sync(0xffffffffu, b1 ? k2[0] : k2[1], 2);
    k1 += __shfl_xor_sync(0xffffffffu, k1, 1);
    const int k = k0 + ((lane >> 1) & 15);
    if ((lane & 1) == 0 && k < K) out[k] = k1;
  }
}

// ---- the same sums as a one-hot GEMM on the tensor cores (16-bit features, hw % 32 == 0, D % 16 == 0, K <= 8 NT) -----
// partial[b][c][k] = sum_p feat[b][c][p] * [label(p) == k]: per warp a [16 channels x pixels] x [pixels x 8 NT classes]
// product with mma.sync.m16n8k16 -- features as row-major A fragments straight from NCHW (two 16-byte loads of 8
// consecutive pixels of rows g and g + 8 per lane), one-hot B fragments made in registers from the lane's own 8 labels
// (narrowed to bytes, 0xff = outside [0, K)), fp32 accumulators in registers: no shared-memory table, no per-class warp
// sums.  Same construction as proto_accumulate_mma_kernel (prototypes.cu) with classes instead of tasks.
constexpr int kSumMmaWarps = 2;
template <typename T>
__device__ __forceinline__ void cs_mma_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                             uint32_t b1) {
  if constexpr (DT<T>::id == BACS_BF16)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <typename T, int NT>
__global__ void __launch_bounds__(32 * kSumMmaWarps) class_sums_mma_kernel(const T* __restrict__ feat, int D, int hw,
                                                                           const int64_t* __restrict__ labels, int K,
                                                                           float* __restrict__ partial) {
  static_assert(sizeof(T) == 2, "16-bit tensor-core operands");
  constexpr uint32_t kOne = DT<T>::id == BACS_BF16 ? 0x3F803F80u : 0x3C003C00u;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int cb = (blockIdx.x * kSumMmaWarps + wid) * 16;
  if (cb >= D) return;
  const int g = lane >> 2, tig = lane & 3;
  const T* rowA = feat + ((int64_t)b * D + cb + g) * hw + tig * 8;
  const T* rowB = rowA + (int64_t)8 * hw;
  const int64_t* lab = labels + (int64_t)b * hw + tig * 8;
  float d[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
  constexpr int U = 2;  // 32-pixel chunks in flight per lane
  for (int q0 = 0; q0 < hw; q0 += 32 * U) {
    uint4 ra[U], rb[U];
    longlong2 l2[U][4];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u * 32;
      if (q < hw) {
        ra[u] = __ldg(reinterpret_cast<const uint4*>(rowA + q));
        rb[u] = __ldg(reinterpret_cast<const uint4*>(rowB + q));
#pragma unroll
        for (int k = 0; k < 4; ++k) l2[u][k] = __ldg(reinterpret_cast<const longlong2*>(lab + q) + k);
      } else {
        ra[u] = rb[u] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int k = 0; k < 4; ++k) l2[u][k] = make_longlong2(-1, -1);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      // the lane's 8 labels as bytes (0xff: outside [0, K))
      uint32_t tw[2] = {0u, 0u};
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const long long l = (e & 1) ? l2[u][e >> 1].y : l2[u][e >> 1].x;
        const uint32_t byte = (l >= 0 && l < K) ? (uint32_t)l : 0xffu;
        tw[e >> 2] |= byte << (8 * (e & 3));
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint32_t a0 = j ? ra[u].z : ra[u].x, a1 = j ? rb[u].z : rb[u].x;
        const uint32_t a2 = j ? ra[u].w : ra[u].y, a3 = j ? rb[u].w : rb[u].y;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const uint32_t m = __vcmpeq4(tw[j], (uint32_t)(8 * nt + g) * 0x01010101u);
          cs_mma_16816<T>(d[nt], a0, a1, a2, a3, __byte_perm(m, 0u, 0x1100) & kOne, __byte_perm(m, 0u, 0x3322) & kOne);
        }
      }
    }
  }
  // D fragment: d[nt][0..1] = (row g, classes 8 nt + 2 tig + {0,1}), d[nt][2..3] = (row g + 8, same classes)
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = 8 * nt + 2 * tig + (e & 1), c = cb + g + (e >> 1) * 8;
      if (k < K) partial[((int64_t)b * D + c) * K + k] = d[nt][e];
    }
  }
}

// sums[k][c] = sum_b partial[b][c][k] (fp64, images in order: deterministic)
__global__ void __launch_bounds__(256) class_sums_finalize_kernel(const float* __restrict__ partial, int B, int D, int K,
                                                                  double* __restrict__ sums) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over (c, k): consecutive threads -> consecutive k
  if (i >= (int64_t)D * K) return;
  const int c = (int)(i / K), k = (int)(i - (int64_t)c * K);
  double s = 0.0;
  for (int b = 0; b < B; ++b) s += (double)partial[((int64_t)b * D + c) * K + k];
  sums[(int64_t)k * D + c] = s;
}

}  // namespace cd
}  // namespace bacs

using namespace bacs;

typedef CUresult (*CdEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static CdEncodeFn cd_encode_fn() {
  static CdEncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<CdEncodeFn>(ptr);
    (void)cudaGetLastError();
  }
  return fn;
}

extern "C" {

size_t bacs_class_distance_workspace_bytes(int32_t B, int32_t Kc, int32_t D, int32_t h, int32_t w) {
  if (B <= 0 || Kc <= 0 || D <= 0 || h <= 0 || w <= 0) return 0;
  return 256;   // the kernel keeps everything on chip; a non-zero size keeps callers' allocation paths uniform
}

int bacs_class_distance(const void* features, int dtype, int32_t B, int32_t D, int32_t h, int32_t w, const void* protos,
                        int32_t Kc, float* dist2, int64_t* nearest, void* workspace, size_t workspace_bytes,
                        bacs_stream_t stream) {
  (void)workspace;
  (void)workspace_bytes;
  BACS_REQUIRE(features && protos && dist2, "bacs_class_distance: null pointer");
  BACS_REQUIRE(dtype == BACS_BF16, "bacs_class_distance: bf16 features and prototypes only (tensor-core operands)");
  BACS_REQUIRE(B > 0 && D > 0 && h > 0 && w > 0 && Kc > 0 && Kc <= 256, "bacs_class_distance: bad shape (Kc <= 256)");
  BACS_REQUIRE(D % 8 == 0 && (h * w) % 8 == 0, "bacs_class_distance: D and h*w must be multiples of 8 (16-byte rows)");
  BACS_REQUIRE((reinterpret_cast<uintptr_t>(protos) & 15) == 0 && (reinterpret_cast<uintptr_t>(features) & 15) == 0,
               "bacs_class_distance: features and prototypes must be 16-byte aligned");
  cd::Params P;
  P.feat = reinterpret_cast<const __nv_bfloat16*>(features);
  P.protos = reinterpret_cast<const __nv_bfloat16*>(protos);
  P.dist2 = dist2;
  P.nearest = nearest;
  P.B = B;
  P.D = D;
  P.Dp = (D + 15) / 16 * 16;
  P.hw = h * w;
  P.Kc = Kc;
  P.Np = (Kc + 31) / 32 * 32;   // a multiple of 8 accumulator columns for each of the four builder warpgroups
  P.tiles_per_image = (P.hw + cd::kTileM - 1) / cd::kTileM;
  P.n_tiles = P.tiles_per_image * B;
  // ring depth: 8 or 4 boxes (a multiple of the four builder warpgroups), whatever fits next to the prototypes
  int stages = cd::kMaxStages;
  if (cd::smem_bytes(P.Np, P.Dp, stages) > (size_t)224 * 1024) stages = 4;
  const size_t smem = cd::smem_bytes(P.Np, P.Dp, stages);
  if (P.Dp > cd::kMaxChunks * cd::kChunkK || smem > (size_t)224 * 1024) {
    set_error("bacs_class_distance: D=%d, Kc=%d do not fit one SM (D <= 512 and the bf16 prototypes, padded to %d x %d, "
              "+ 32 KB of staging <= 224 KB of shared memory)", D, Kc, P.Np, P.Dp);
    return BACS_ERR_UNSUPPORTED;
  }
  P.stages = stages;
  CdEncodeFn enc = cd_encode_fn();
  if (!enc) {
    set_error("bacs_class_distance: cuTensorMapEncodeTiled is not available from this driver");
    return BACS_ERR_UNSUPPORTED;
  }
  CUtensorMap map;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)P.hw, (cuuint64_t)D, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)P.hw * 2, (cuuint64_t)P.hw * 2 * (cuuint64_t)D};
    const cuuint32_t box[3] = {(cuuint32_t)cd::kTileM, (cuuint32_t)cd::kChunkK, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(features), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("bacs_class_distance: cuTensorMapEncodeTiled failed (%d)", (int)r);
      return BACS_ERR_CUDA;
    }
  }
  cudaError_t e = cudaFuncSetAttribute(cd::class_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("bacs_class_distance: shared memory opt-in failed: %s", cudaGetErrorString(e));
    return BACS_ERR_CUDA;
  }
  const int grid = std::min(P.n_tiles, sm_count());
  cd::class_distance_kernel<<<grid, cd::kThreads, smem, (cudaStream_t)stream>>>(map, P);
  BACS_CHECK_LAUNCH("bacs_class_distance");
  return BACS_OK;
}

size_t bacs_class_sums_workspace_bytes(int32_t B, int32_t D, int32_t K) {
  if (B <= 0 || D <= 0 || K <= 0) return 0;
  return align_up((size_t)B * D * K * sizeof(float), 256);
}

int bacs_class_sums(const void* features, int dtype, int32_t B, int32_t D, int32_t h, int32_t w, const int64_t* labels_down,
                    int32_t K, double* sums, void* workspace, size_t workspace_bytes, bacs_stream_t stream) {
  BACS_REQUIRE(features && labels_down && sums && workspace, "bacs_class_sums: null pointer");
  BACS_REQUIRE(B > 0 && B < 65536 && D > 0 && h > 0 && w > 0 && K > 0 && K <= 1024, "bacs_class_sums: bad shape (K <= 1024)");
  if (workspace_bytes < bacs_class_sums_workspace_bytes(B, D, K)) {
    set_error("bacs_class_sums: workspace %zu < %zu", workspace_bytes, bacs_class_sums_workspace_bytes(B, D, K));
    return BACS_ERR_WORKSPACE;
  }
  // warps (= channel rows) per block: as many [K][32] tables as fit 200 KB of shared memory, at most 8
  int warps = (int)std::min<size_t>(cd::kSumWarps, (size_t)200 * 1024 / ((size_t)K * 32 * sizeof(float)));
  BACS_REQUIRE(warps >= 1, "bacs_class_sums: K=%d does not fit a shared-memory table", K);
  const size_t smem = (size_t)warps * K * 32 * sizeof(float);
  float* partial = reinterpret_cast<float*>(workspace);
  cudaStream_t s = (cudaStream_t)stream;
  dim3 grid((D + warps - 1) / warps, B);
  // 16-bit features on 32-pixel chunks, K <= 160 (ADE20K's 151): one-hot GEMM on the tensor cores (BACS_NO_SUMS_MMA=1: off)
  const bool mma = dtype != BACS_F32 && (h * w) % 32 == 0 && D % 16 == 0 && K <= 160 &&
                   (reinterpret_cast<uintptr_t>(features) & 15) == 0 && (reinterpret_cast<uintptr_t>(labels_down) & 15) == 0 &&
                   getenv("BACS_NO_SUMS_MMA") == nullptr;
  if (mma) {
    dim3 mgrid((D / 16 + cd::kSumMmaWarps - 1) / cd::kSumMmaWarps, B);
    const int nt = (K + 7) / 8;
#define BACS_CS_LAUNCH(TT, NTV)                                                                                  \
  cd::class_sums_mma_kernel<TT, NTV><<<mgrid, 32 * cd::kSumMmaWarps, 0, s>>>(reinterpret_cast<const TT*>(features), D, \
                                                                               h * w, labels_down, K, partial)
#define BACS_CS_NT(TT)                          \
  do {                                          \
    if (nt <= 4) BACS_CS_LAUNCH(TT, 4);         \
    else if (nt <= 8) BACS_CS_LAUNCH(TT, 8);    \
    else if (nt <= 12) BACS_CS_LAUNCH(TT, 12);  \
    else if (nt <= 16) BACS_CS_LAUNCH(TT, 16);  \
    else BACS_CS_LAUNCH(TT, 20);                \
  } while (0)
    if (dtype == BACS_BF16) BACS_CS_NT(__nv_bfloat16);
    else BACS_CS_NT(__half);
#undef BACS_CS_NT
#undef BACS_CS_LAUNCH
  } else {
  BACS_DISPATCH_DTYPE(dtype, TT, {
    auto kern = cd::class_sums_kernel<TT>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) {
        set_error("bacs_class_sums: shared memory opt-in failed: %s", cudaGetErrorString(e));
        return BACS_ERR_CUDA;
      }
    }
    const int vec = ((h * w) % 8 == 0 && (reinterpret_cast<uintptr_t>(features) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(labels_down) & 15) == 0) ? 1 : 0;
    kern<<<grid, 32 * cd::kSumWarps, smem, s>>>(reinterpret_cast<const TT*>(features), D, h * w, labels_down, K, warps, vec,
                                                 partial);
  });
  }
  BACS_CHECK_LAUNCH("bacs_class_sums");
  const int64_t n = (int64_t)D * K;
  cd::class_sums_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(partial, B, D, K, sums);
  BACS_CHECK_LAUNCH("bacs_class_sums(finalize)");
  return BACS_OK;
}

}  // extern "C"
