// Large class counts in 16-bit storage (64 <= K <= 152: ADE20K's 151 in bf16 / fp16): the per-pixel loss in ONE pass
// over the logits, the [K] x 2-pixel column of a pixel pair held in the registers of TWO lanes.
//
// The two streaming passes of pixel_stream.cuh read every logit twice (3 K s bytes per pixel against the algorithmic
// 2 K s).  Here a CTA of four warps owns 128-pixel tiles.  Lanes l and l + 16 of a warp share one pair of adjacent
// pixels: lane l keeps channels 0 .. 75 of the pair, lane l + 16 channels 76 .. 151, one 32-bit register per channel
// holding the packed pair exactly as it sits in memory (76 registers -> 128 registers per thread, 16 warps per SM; a
// whole column per thread needs 255 registers, leaves two warps per scheduler and stalls on its own dependent
// instructions: 1.18 ms).
//   load      one 3-D tensor-map TMA box [K][128] (38.6 KB at K = 151) per tile into the CTA's single landing buffer;
//             the threads copy their half column into registers (LDS.32 with immediate offsets), the CTA synchronises and
//             the box of the CTA's NEXT tile is requested at once -- it lands while this tile is computed from the
//             registers, so the registers are the second pipeline stage and no warp waits on a cold load.  (First
//             version: K independent 4-byte global loads per thread, 128 bytes per warp request: 957 us for the
//             forward alone -- the SM's queue of outstanding L1 requests, not HBM, was the limit.)
//   max       running max / first arg-max on the packed words (HMNMX2 + HSET2 + LOP3 per channel, as the tile kernels),
//             combined across the two lanes by shuffles (ties -> the lower channel half);
//   sums      exponent sums against the final max (no online rescaling), eight channels at a time; a block that lies
//             below old_cl is also added to the old classes' sum; the up to seven old channels of the block the boundary
//             falls into are added from memory by a short rolled loop; the lanes exchange their partial sums;
//   terms     lane l evaluates the pair's first pixel, lane l + 16 the second, with the same stream_pixel_stage() /
//             pixel_terms() as the streaming kernel (labels, seen probability, loss terms, distill mask, focal
//             gradient, arg-max); the gradient coefficients are exchanged by shuffles;
//   gradient  e_k * cg[group(k)] - [k==0] d0 from the registers (second ex2 per logit; keeping the exponentials would
//             take another register per channel and pixel), packed and stored with the coefficient of the block's
//             group; the old channels of the boundary block and the label's own channel (-dy applied before the
//             rounding to the storage type, as in the streaming gradient pass) are then re-stored.
// HBM traffic: 2 K s + 17 bytes per pixel.
#pragma once
#include "pixel_stream.cuh"

namespace bacs {

constexpr int kRegsKH = 76;      // channel registers of a thread; K <= 2 * kRegsKH
constexpr int kRegsKMax = 2 * kRegsKH;
constexpr int kRegsNT = 128;     // threads of a CTA = pixels of a tile
constexpr int kRegsCTAs = 4;     // resident CTAs per SM (DESIGN 5.1a)

struct alignas(64) RegsParams {
  CUtensorMap tmap_in;  // logits as (H*W, K, B), box (NT, K, 1)
  StreamParams s;       // s.coef != nullptr <=> a gradient is wanted; one partial row per CTA
  int tiles_per_image;
  int n_tiles;          // B * tiles_per_image, walked with stride gridDim.x
};

template <typename T> struct RegsNegInf;
template <> struct RegsNegInf<__nv_bfloat16> { static constexpr uint32_t pair = 0xff80ff80u; };
template <> struct RegsNegInf<__half> { static constexpr uint32_t pair = 0xfc00fc00u; };

template <typename T>
__device__ __forceinline__ uint32_t regs_pack(F2 v) {
  if constexpr (DT<T>::id == BACS_BF16) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(f2lo(v), f2hi(v));
    return *reinterpret_cast<const uint32_t*>(&h);
  } else {
    const __half2 h = __floats2half2_rn(f2lo(v), f2hi(v));
    return *reinterpret_cast<const uint32_t*>(&h);
  }
}

// NT threads = NT pixels per tile (NT / 2 pixel pairs x 2 lanes) = one TMA box row; MINB CTAs per SM
// (max, first arg-max) of two disjoint channel sets of the same pixel pair; ties -> the lower channel index
template <typename T>
__device__ __forceinline__ void regs_merge_max(typename Raw<T>::Max& a, const typename Raw<T>::Max& b) {
  const uint32_t take = __hgt2_mask(b.m, a.m) | (__heq2_mask(b.m, a.m) & __vcmpltu2(b.a, a.a));
  a.m = __hmax2(b.m, a.m);
  a.a = (a.a & ~take) | (b.a & take);
}

template <typename T, int KH, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) pixel_regs_kernel(const __grid_constant__ RegsParams q) {
  constexpr int kRegsThreads = NT, kRegsTile = NT;
  static_assert(sizeof(T) == 2 && KH % 4 == 0, "packed pixel pairs of a 16-bit type, channel blocks of 8 (+ one of 4)");
  extern __shared__ __align__(128) unsigned char regs_smem[];  // landing buffer [K][NT] T, then [7][NT] boundary words
  __shared__ uint32_t fix_words[7 * NT];
  __shared__ uint64_t bar_full;
  __shared__ float red_scratch[kStreamThreads / 32][BACS_NACC];
  __shared__ float s_norm_sh;
  using R = Raw<T>;
  constexpr unsigned kFull = 0xffffffffu;
  const StreamParams& p = q.s;
  const bacs_pixel_args& a = p.a;
  const int tid = threadIdx.x, lane = tid & 31;
  const int half = lane >> 4;                        // which channel half, and which pixel of the pair in the terms
  const int pr = (tid >> 5) * 16 + (lane & 15);      // pixel pair of the tile
  const int hb = half * KH;                          // first channel of this lane
  const int K = a.K;
  const uint32_t box_bytes = (uint32_t)K * kRegsTile * sizeof(T);
  auto request = [&](int t) {  // thread 0: the box of tile t
    const int tb = t / q.tiles_per_image, ti = t - tb * q.tiles_per_image;
    mbar_expect_tx(&bar_full, box_bytes);
    tma_load_3d(regs_smem, &q.tmap_in, ti * kRegsTile, 0, tb, &bar_full);
  };
  int tile = (int)blockIdx.x;
  if (tid == 0) {
    mbar_init(&bar_full, 1);
    fence_mbar_init();
    if (tile < q.n_tiles) request(tile);
  }
  const float s_norm = stream_norm(p, &s_norm_sh);  // (contains the barrier that publishes bar_full)
  float acc[BACS_NACC];
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) acc[i] = 0.f;
  const int64_t HW = (int64_t)a.H * a.W;
  const int old_cl = min(max(a.old_cl, 0), K);
  const bool have_seen = (a.z != nullptr) || (a.seen_max != nullptr);
  const F2 l2e2 = f2b(kLog2e);
  const uint32_t* col = reinterpret_cast<const uint32_t*>(regs_smem) + hb * (kRegsTile / 2) + pr;  // + i * 128 words
  // the old channels of the block of this lane that the old / new boundary falls into: [fix_lo, fix_hi)
  const int fix_lo = max(hb + ((old_cl - hb) & ~7), 1), fix_hi = (old_cl > hb && old_cl < hb + KH) ? old_cl : 0;

  // label and seen-head taps of this lane's pixel of tile t into L1 (the terms of that tile then find them there)
  auto prefetch_side = [&](int t) {
    const int tb = t / q.tiles_per_image;
    const int64_t pix = (int64_t)(t - tb * q.tiles_per_image) * kRegsTile + 2 * pr + half;
    asm volatile("prefetch.global.L1 [%0];" ::"l"(a.labels + (int64_t)tb * HW + pix));
    if (a.z) {
      const int Y = (int)(pix / a.W), X = (int)(pix - (int64_t)Y * a.W);
      const Lerp ly = lerp_align_corners(Y, a.h, p.sy), lx = lerp_align_corners(X, a.w, p.sx);
      const float* zb = a.z + (int64_t)tb * a.T * a.h * a.w;
      for (int t2 = 0; t2 < a.T; ++t2) {
        const float* zt = zb + (int64_t)t2 * a.h * a.w;
        asm volatile("prefetch.global.L1 [%0];" ::"l"(zt + ly.i0 * a.w + lx.i0));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(zt + ly.i1 * a.w + lx.i1));
      }
    }
  };
  if (tile < q.n_tiles) prefetch_side(tile);

  for (uint32_t it = 0; tile < q.n_tiles; tile += (int)gridDim.x, ++it) {
    const int b = tile / q.tiles_per_image;
    const int64_t p0 = (int64_t)(tile - b * q.tiles_per_image) * kRegsTile + 2 * pr;  // the pair's first pixel
    const T* base = reinterpret_cast<const T*>(a.logits) + (int64_t)b * K * HW + p0;
    uint32_t w[KH];
    const long long my_lab = __ldg(a.labels + (int64_t)b * HW + p0 + half);
    if (tile + (int)gridDim.x < q.n_tiles) prefetch_side(tile + (int)gridDim.x);
    // ---- landing buffer -> registers; then the buffer is free for the CTA's next tile ------------------------------
    mbar_wait(&bar_full, it & 1u);
    auto load_column = [&]() {
#pragma unroll
      for (int c0 = 0; c0 < KH; c0 += 8) {
        if (KH + c0 + 8 <= K) {  // (uniform) the block exists in both lanes' halves
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (c0 + i < KH) w[c0 + i] = col[(c0 + i) * (kRegsTile / 2)];
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (c0 + i < KH) w[c0 + i] = (hb + c0 + i < K) ? col[(c0 + i) * (kRegsTile / 2)] : RegsNegInf<T>::pair;
        }
      }
    };
    load_column();
    float my_xy = 0.f;  // the label's own logit
    if (my_lab >= 0 && my_lab < K)
      my_xy = DT<T>::to_f(reinterpret_cast<const T*>(regs_smem)[(int)my_lab * kRegsTile + 2 * pr + half]);
    // ---- max / first arg-max (channels >= K hold -inf and never win) ---------------------------------------------
    float m[2];
    int am[2];
    {
      // two independent running maxima (even / odd channels) halve the dependent HMNMX2 -> HSET2 chain
      typename R::Max mt = R::init(w[0]), mu = R::init(w[1]);
      R::set_first(mt, 0);
      R::set_first(mu, 1);
#pragma unroll
      for (int i = 2; i < KH; ++i) {
        if (i & 1) R::update(mu, w[i], i);
        else R::update(mt, w[i], i);
      }
      regs_merge_max<T>(mt, mu);
      R::finish(mt, m[0], m[1], am[0], am[1]);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float om = __shfl_xor_sync(kFull, m[j], 16);
        const int oa = __shfl_xor_sync(kFull, am[j], 16) + (KH - hb);  // the other lane's first channel is KH - hb
        const int ma = am[j] + hb;
        const bool other = half ? (om >= m[j]) : (om > m[j]);  // ties go to the lower channel half
        m[j] = fmaxf(m[j], om);
        am[j] = other ? oa : ma;
      }
    }
    const F2 nm2 = f2(-m[0] * kLog2e, -m[1] * kLog2e);
    auto expo_at = [&](uint32_t word, F2 nm) {
      float v0, v1;
      R::unpack(word, v0, v1);
      const F2 arg = fma2(f2(v0, v1), l2e2, nm);
      return f2(ex2_fast(f2lo(arg)), ex2_fast(f2hi(arg)));
    };
    auto expo = [&](uint32_t word) { return expo_at(word, nm2); };
    // ---- exponent sums: all foreground channels, and the old ones (1 <= c < old_cl) ------------------------------
    float so[2], sn[2];
    {
      F2 s2 = f2b(0.f), so2 = f2b(0.f);
#pragma unroll
      for (int c0 = 0; c0 < KH; c0 += 8) {
        const int bw = c0 + 8 <= KH ? 8 : KH - c0;
        // the eight exponentials of a block are independent values summed as a tree: written as one running sum the
        // compiler reuses one register pair per channel and every ex2 waits for the add before it (IPC 0.65 per scheduler)
        F2 e[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) e[i] = i < bw ? expo(w[c0 + i]) : f2b(0.f);
        if (c0 == 0) e[0] = hb ? e[0] : f2b(0.f);  // the background channel is not part of the sums
        const F2 t = add2(add2(add2(e[0], e[1]), add2(e[2], e[3])), add2(add2(e[4], e[5]), add2(e[6], e[7])));
        s2 = add2(s2, t);
        if (hb + c0 + bw <= old_cl) so2 = add2(so2, t);
      }
      for (int c = fix_lo; c < fix_hi; ++c)  // the old channels of the boundary block (at most seven)
        so2 = add2(so2, expo(reinterpret_cast<const uint32_t*>(regs_smem)[c * (kRegsTile / 2) + pr]));
      so[0] = f2lo(so2) + __shfl_xor_sync(kFull, f2lo(so2), 16);
      so[1] = f2hi(so2) + __shfl_xor_sync(kFull, f2hi(so2), 16);
      sn[0] = f2lo(s2) + __shfl_xor_sync(kFull, f2lo(s2), 16) - so[0];  // only so + sn (= the total to an ulp) is used
      sn[1] = f2hi(s2) + __shfl_xor_sync(kFull, f2hi(s2), 16) - so[1];
    }
    // ---- per-pixel terms: this lane evaluates pixel `half` of the pair ---------------------------------------------
    float cgA[2], cgB[2], cgC[2], d0[2];  // per pixel of the pair: coefficient of channel 0 / old / new classes, d0
    float my_dy = 0.f;
    int my_y = 0;
    {
      float x0[2];
      R::unpack(w[0], x0[0], x0[1]);                      // (channel 0 lives in the lower lane)
      const float x0_hi = __shfl_xor_sync(kFull, x0[1], 16);
      const float m1[1] = {half ? m[1] : m[0]}, so1[1] = {half ? so[1] : so[0]}, sn1[1] = {half ? sn[1] : sn[0]};
      const float x01[1] = {half ? x0_hi : x0[0]};
      const int am1[1] = {half ? am[1] : am[0]};
      float c0v = 0.f, c1v = 0.f, c2v = 0.f, d0v = 0.f;
      stream_pixel_stage<T, 1, true>(p, b, s_norm, old_cl, have_seen, p0 + half, base + half, m1, so1, sn1, x01, am1, acc,
                                     [&](int, float, const PixCoef& pc, long long l) {
                                       c0v = pc.cg0; c1v = pc.cg1; c2v = pc.cg2; d0v = pc.d0;
                                       my_dy = pc.dy;
                                       my_y = (int)l;
                                     }, my_lab, my_xy);
      const float o0 = __shfl_xor_sync(kFull, c0v, 16), o1 = __shfl_xor_sync(kFull, c1v, 16);
      const float o2 = __shfl_xor_sync(kFull, c2v, 16), o3 = __shfl_xor_sync(kFull, d0v, 16);
      cgA[0] = half ? o0 : c0v; cgA[1] = half ? c0v : o0;
      cgB[0] = half ? o1 : c1v; cgB[1] = half ? c1v : o1;
      cgC[0] = half ? o2 : c2v; cgC[1] = half ? c2v : o2;
      d0[0] = half ? o3 : d0v;  d0[1] = half ? d0v : o3;
    }
    // ---- the column a second time (it is not kept across the terms: 76 + their ~80 registers would spill), then the
    //      landing buffer is free for the CTA's next tile, which lands during the gradient pass
    asm volatile("" ::: "memory");
    if (a.dlogits) {
      load_column();
      for (int c = fix_lo; c < fix_hi; ++c)
        fix_words[(c - fix_lo) * NT + tid] = reinterpret_cast<const uint32_t*>(regs_smem)[c * (kRegsTile / 2) + pr];
    }
    __syncthreads();
    if (tid == 0 && tile + (int)gridDim.x < q.n_tiles) request(tile + (int)gridDim.x);
    if (!a.dlogits) continue;  // (uniform over the grid)
    // ---- gradient ----------------------------------------------------------------------------------------------------
    T* gbase = reinterpret_cast<T*>(a.dlogits) + (int64_t)b * K * HW + p0;
    const F2 c0_2 = f2(cgA[0], cgA[1]), c1_2 = f2(cgB[0], cgB[1]), c2_2 = f2(cgC[0], cgC[1]);
    const F2 nd0_2 = f2(-d0[0], -d0[1]);
    {
      // the exponentials are taken a second time: an opaque copy of -max*log2e keeps the compiler from carrying the
      // 2 x KH values of the sums pass across the terms (they would be spilled)
      F2 nm2g = nm2;
      asm volatile("" : "+l"(nm2g.v));
      auto expo = [&](uint32_t word) { return expo_at(word, nm2g); };
      uint32_t* gp = reinterpret_cast<uint32_t*>(gbase + (int64_t)hb * HW);
      const int64_t gstep = HW / 2;  // words per channel row
#pragma unroll
      for (int c0 = 0; c0 < KH; c0 += 8) {
        const int bw = c0 + 8 <= KH ? 8 : KH - c0;
        const bool blk_old = hb + c0 + bw <= old_cl;
        const F2 cg = blk_old ? c1_2 : c2_2;
        uint32_t out[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (i < bw) {
            const F2 e = expo(w[c0 + i]);
            F2 g = mul2(e, cg);
            if (c0 + i == 0) g = hb ? g : fma2(e, c0_2, nd0_2);
            out[i] = regs_pack<T>(g);
          }
        }
        if (KH + c0 + bw <= K) {  // (uniform) the block exists in both lanes' halves
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (i < bw) gp[(c0 + i) * gstep] = out[i];
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (i < bw && hb + c0 + i < K) gp[(c0 + i) * gstep] = out[i];
        }
      }
    }
    // the old channels of the boundary block were written with the new classes' coefficient
    for (int c = fix_lo; c < fix_hi; ++c) {
      const F2 e = expo(fix_words[(c - fix_lo) * NT + tid]);
      *reinterpret_cast<uint32_t*>(gbase + (int64_t)c * HW) = regs_pack<T>(mul2(e, c1_2));
    }
    __syncwarp();  // the label's channel may have been written by the other lane of the pair
    // the label's own channel: recomputed in fp32 so that -dy is applied before the rounding to the storage type
    if (my_dy != 0.f) {
      const int y = my_y;
      const float e = ex2_fast(fmaf(my_xy, kLog2e, -(half ? m[1] : m[0]) * kLog2e));
      const float cg = y == 0 ? (half ? cgA[1] : cgA[0]) : (y < old_cl ? (half ? cgB[1] : cgB[0]) : (half ? cgC[1] : cgC[0]));
      gbase[(int64_t)y * HW + half] = DT<T>::from_f(e * cg - my_dy - (y == 0 ? (half ? d0[1] : d0[0]) : 0.f));
    }
  }
  stream_flush_acc(p, acc, red_scratch, (int64_t)blockIdx.x, kRegsThreads / 32);
}

}  // namespace bacs
