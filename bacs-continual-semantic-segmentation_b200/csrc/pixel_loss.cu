// The fused per-pixel kernel of the BACS loss step.
//
// Persistent, warp-specialised CTAs (one producer warp + 8 consumer warps).  A tile is P
// consecutive pixels of one image; its K logit rows ([K][P], NCHW so every row is one
// contiguous segment) travel global -> shared memory by 1-D TMA bulk copies
// (cp.async.bulk + mbarrier) through a ring of stages.  Consumers pull the tile into
// registers, compute the softmax statistics ONCE per pixel and derive from them, in the
// same pass:
//   * background-aware unbiased CE  (training/loss_utils.py:542-585)   mode WEIGHTED_CE
//   * plain / class-weighted CE     (loss/base_loss.py:237-240)        mode CE
//   * MiB unbiased CE               (training/loss_utils.py:492-520)   mode UNBIASED_CE
//   * per-image importance score    (loss/bacs_loss.py:183-189)        mode SCORE
//   * seen-detector focal loss of one head + its gradient w.r.t. the low-res head output
//     (loss/base_loss.py:255-272, smp FocalLoss binary; bilinear x16 align_corners=True
//      evaluated on the fly, networks/bg_detector.py:13-15)
//   * the teacher-distill pixel mask (loss/bacs_loss.py:282-285)
//   * arg-max (loss/bacs_loss.py:255)
// The gradient rows overwrite the logits of the stage in place and leave through TMA bulk
// stores issued by the producer warp, so HBM sees one read and one write of [B,K,H,W]
// plus 8 + 8 (+1) bytes per pixel, and the consumers never wait for a store.
#include <algorithm>
#include <cstdlib>

#include "pixel_fast.cuh"  // Raw<T>: packed pixel pairs

namespace bacs {

// Shared-memory layout (dynamic): [stages][K*PITCH] tiles | zr[T][w] | gacc[w+1]
// COOP (large K, one pixel per thread for everything per-pixel): the two threads of an even/odd lane pair walk the
// channel loops together on their two adjacent pixels as PACKED pairs, each taking every other channel, and
// exchange max / arg-max / sums / coefficients by shuffle.  Rows are 64 bytes longer than P elements so that the
// two halves of a warp (rows c and c+1) hit disjoint banks.
template <typename T, int PPT, bool ROWTILE, bool COOP = false>
__global__ void __launch_bounds__(kConsumers + 32, PPT == 1 ? 2 : 1) pixel_loss_kernel(const PixelParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t bar_full[kMaxStages];  // producer -> consumers: tile landed
  __shared__ uint64_t bar_done[kMaxStages];  // consumers -> producer: gradients written; store / refill the stage
  __shared__ float red_scratch[kConsumerWarps][BACS_NACC];
  __shared__ float s_norm_sh;

  const bacs_pixel_args& a = p.a;
  const int P = p.P, K = a.K, S = p.stages;
  const int PITCH = COOP ? P + 64 / (int)sizeof(T) : P;  // elements between channel rows of a tile
  const int tid = threadIdx.x;
  const int64_t HW = (int64_t)a.H * a.W;
  const size_t tile_elems = (size_t)K * PITCH;
  T* tiles = reinterpret_cast<T*>(smem_raw);
  float* zr = reinterpret_cast<float*>(smem_raw + ((S * tile_elems * sizeof(T) + 15) / 16) * 16);
  float* gacc = zr + (ROWTILE ? a.T * a.w : 0);
  const int my_tiles = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  // k-th tile of this CTA: image b, first pixel p0, npx pixels
  auto tile_geom = [&](int k, int& b, int64_t& p0, int& npx) {
    const int tile = (int)blockIdx.x + k * (int)gridDim.x;
    b = tile / p.tiles_per_image;
    p0 = (int64_t)(tile - b * p.tiles_per_image) * P;
    npx = (int)min((int64_t)P, HW - p0);
  };

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_done[s], kConsumers);
    }
    fence_mbar_init();
    s_norm_sh = 0.f;
  }
  __syncthreads();
  // CE-type modes: gradient normaliser from the label histogram (device-side, no host sync)
  if (tid < 32 && a.mode != BACS_PIX_WEIGHTED_CE && a.dlogits != nullptr) {
    double s = 0.0;
    for (int c = tid; c < K && c < 256; c += 32)
      if (c != a.ignore_index)
        s += (double)a.hist[c] * ((a.mode == BACS_PIX_CE && a.class_w) ? (double)a.class_w[c] : 1.0);
    s = warp_sum(s);
    if (tid == 0) s_norm_sh = s > 0.0 ? (float)(1.0 / s) : 0.f;
  }
  __syncthreads();

  // =====================================================================================
  // producer warp
  // =====================================================================================
  if (tid >= kConsumers) {
    const int lane = tid - kConsumers;
    auto load_tile = [&](int k) {
      int b, npx;
      int64_t p0;
      tile_geom(k, b, p0, npx);
      const int s = k % S;
      T* dst = tiles + (size_t)s * tile_elems;
      const T* src = reinterpret_cast<const T*>(a.logits) + (int64_t)b * K * HW + p0;
      const bool bulk = p.use_bulk && ((npx * (int)sizeof(T)) & 15) == 0;
      if (bulk) {
        if (lane == 0) mbar_expect_tx(&bar_full[s], (uint32_t)(K * npx * (int)sizeof(T)));
        __syncwarp();
        for (int c = lane; c < K; c += 32)
          bulk_g2s(dst + (size_t)c * PITCH, src + (int64_t)c * HW, (uint32_t)(npx * sizeof(T)), &bar_full[s]);
      } else {  // ragged / unaligned rows: plain copies by the producer warp
        for (int c = 0; c < K; ++c)
          for (int i = lane; i < npx; i += 32) dst[(size_t)c * PITCH + i] = src[(int64_t)c * HW + i];
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_full[s]);
      }
    };
    const int pre = min(S, my_tiles);
    for (int k = 0; k < pre; ++k) load_tile(k);
    for (int k = 0; k < my_tiles; ++k) {
      const int s = k % S;
      mbar_wait(&bar_done[s], (uint32_t)((k / S) & 1));
      if (a.dlogits) {
        int b, npx;
        int64_t p0;
        tile_geom(k, b, p0, npx);
        const T* src = tiles + (size_t)s * tile_elems;
        T* dst = reinterpret_cast<T*>(a.dlogits) + (int64_t)b * K * HW + p0;
        const bool bulk = p.use_bulk && ((npx * (int)sizeof(T)) & 15) == 0;
        if (bulk) {
          for (int c = lane; c < K; c += 32)
            bulk_s2g(dst + (int64_t)c * HW, src + (size_t)c * PITCH, (uint32_t)(npx * sizeof(T)));
          bulk_commit();
          if (k + S < my_tiles) bulk_wait_read0();  // the stage is about to be refilled
        } else {
          for (int c = 0; c < K; ++c)
            for (int i = lane; i < npx; i += 32) dst[(int64_t)c * HW + i] = src[(size_t)c * PITCH + i];
        }
        __syncwarp();
      }
      if (k + S < my_tiles) load_tile(k + S);
    }
    bulk_wait_all();
    return;
  }

  // =====================================================================================
  // consumer warps
  // =====================================================================================
  const int lane = tid & 31, wid = tid >> 5;
  const int px0 = tid * PPT;
  const int old_cl = min(max(a.old_cl, 0), K);
  const bool have_seen = (a.z != nullptr) || (a.seen_max != nullptr);
  const float s_norm = s_norm_sh;
  float acc[BACS_NACC];
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) acc[i] = 0.f;

  auto load_labels = [&](int k, int64_t* lab) {
    int b, npx;
    int64_t p0;
    tile_geom(k, b, p0, npx);
    const int64_t* src = a.labels + (int64_t)b * HW + p0 + px0;
    if (PPT == 2 && px0 + 1 < npx && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
      const longlong2 v = __ldg(reinterpret_cast<const longlong2*>(src));
      lab[0] = v.x;
      lab[PPT - 1] = v.y;
    } else {
#pragma unroll
      for (int j = 0; j < PPT; ++j) lab[j] = (px0 + j < npx) ? __ldg(src + j) : (int64_t)a.ignore_index;
    }
  };
  int64_t lab_next[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) lab_next[j] = a.ignore_index;
  if (my_tiles > 0) load_labels(0, lab_next);

  for (int k = 0; k < my_tiles; ++k) {
    int b, npx;
    int64_t p0;
    tile_geom(k, b, p0, npx);
    const int s = k % S;
    T* tile = tiles + (size_t)s * tile_elems;
    int64_t lab[PPT];
#pragma unroll
    for (int j = 0; j < PPT; ++j) lab[j] = lab_next[j];
    if (k + 1 < my_tiles) load_labels(k + 1, lab_next);

    // ---- per-pixel side inputs --------------------------------------------------------
    int y[PPT];
    bool is_ign[PPT];
    float seen[PPT], zfoc[PPT], wx1[PPT];
    int cx0[PPT], cdx[PPT];
    int cell[PPT], cell_dy[PPT];  // generic (non row-tile) focal scatter bookkeeping
    float wy1g[PPT];
    int Yrow = 0;
    Lerp ly_row = {0, 0, 0.f};
    if (ROWTILE && a.z) {
      // the tile lies inside image row Yrow: interpolate the T head rows in y once
      Yrow = (int)(p0 / a.W);
      ly_row = lerp_align_corners(Yrow, a.h, p.sy);
      consumer_sync();  // previous tile's readers of zr / gacc are done
      const float* zb = a.z + (int64_t)b * a.T * a.h * a.w;
      const float wy0 = 1.f - ly_row.w1;
      for (int i = tid; i < a.T * a.w; i += kConsumers) {
        const int t = i / a.w, j = i - t * a.w;
        const float* zt = zb + (int64_t)t * a.h * a.w;
        zr[i] = __fadd_rn(__fmul_rn(wy0, __ldg(zt + ly_row.i0 * a.w + j)),
                          __fmul_rn(ly_row.w1, __ldg(zt + ly_row.i1 * a.w + j)));
      }
      if (a.gz)
        for (int i = tid; i < a.w + 1; i += kConsumers) gacc[i] = 0.f;
      consumer_sync();
    }
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      const int px = px0 + j;
      y[j] = -1;
      is_ign[j] = true;
      seen[j] = 0.f;
      zfoc[j] = 0.f;
      wx1[j] = 0.f;
      cx0[j] = -1;
      cdx[j] = 0;
      cell[j] = -1;
      cell_dy[j] = 0;
      wy1g[j] = 0.f;
      if (px < npx) {
        const int64_t l = lab[j];
        if (l == a.ignore_index) {
        } else if (l >= 0 && l < K) {
          y[j] = (int)l;
          is_ign[j] = false;
        } else {
          acc[BACS_ACC_INVALID] += 1.f;
        }
        if (a.seen_max) seen[j] = __ldg(a.seen_max + (int64_t)b * HW + p0 + px);
        if (a.z) {
          const int64_t pix = p0 + px;
          float zmax = -INFINITY;
          if (ROWTILE) {
            const int X = (int)(pix - (int64_t)Yrow * a.W);
            const Lerp lx = lerp_align_corners(X, a.w, p.sx);
            const float wx0 = 1.f - lx.w1;
            for (int t = 0; t < a.T; ++t) {
              const float v = __fadd_rn(__fmul_rn(wx0, zr[t * a.w + lx.i0]), __fmul_rn(lx.w1, zr[t * a.w + lx.i1]));
              zmax = fmaxf(zmax, v);
              if (t == a.focal_head) zfoc[j] = v;
            }
            cx0[j] = lx.i0;
            cdx[j] = lx.i1 - lx.i0;
            wx1[j] = lx.w1;
          } else {
            const int Y = (int)(pix / a.W), X = (int)(pix - (int64_t)Y * a.W);
            const Lerp ly = lerp_align_corners(Y, a.h, p.sy), lx = lerp_align_corners(X, a.w, p.sx);
            const float wx0 = 1.f - lx.w1, wy0 = 1.f - ly.w1;
            const float* zb = a.z + (int64_t)b * a.T * a.h * a.w;
            const int o00 = ly.i0 * a.w + lx.i0, o01 = ly.i0 * a.w + lx.i1;
            const int o10 = ly.i1 * a.w + lx.i0, o11 = ly.i1 * a.w + lx.i1;
            for (int t = 0; t < a.T; ++t) {
              const float* zt = zb + (int64_t)t * a.h * a.w;
              const float left = __fadd_rn(__fmul_rn(wy0, __ldg(zt + o00)), __fmul_rn(ly.w1, __ldg(zt + o10)));
              const float right = __fadd_rn(__fmul_rn(wy0, __ldg(zt + o01)), __fmul_rn(ly.w1, __ldg(zt + o11)));
              const float v = __fadd_rn(__fmul_rn(wx0, left), __fmul_rn(lx.w1, right));
              zmax = fmaxf(zmax, v);
              if (t == a.focal_head) zfoc[j] = v;
            }
            cell[j] = o00;
            cdx[j] = lx.i1 - lx.i0;
            cell_dy[j] = (ly.i1 - ly.i0) * a.w;
            wy1g[j] = ly.w1;
            wx1[j] = lx.w1;
          }
          if (!a.seen_max) seen[j] = sigmoid_fast(zmax);
        }
      }
    }

    // ---- wait for the tile, softmax statistics, gradients ------------------------------
    mbar_wait(&bar_full[s], (uint32_t)((k / S) & 1));
    const bool live = px0 < npx;
    const unsigned live_mask = __ballot_sync(0xffffffffu, live);  // (cooperative path: pairs are live together)
    PixCoef pc[PPT];
    float gfoc[PPT];
    uint8_t dmask[PPT];
    int amax[PPT];
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      gfoc[j] = 0.f;
      dmask[j] = 0;
      amax[j] = 0;
    }
    if (live) {
      T* col = tile + px0;
      float xy[PPT], x0[PPT];
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        xy[j] = (y[j] >= 0) ? DT<T>::to_f(col[(size_t)y[j] * PITCH + j]) : 0.f;
        x0[j] = DT<T>::to_f(col[j]);
      }
      if constexpr (COOP) {
        // ---------------- cooperative packed path (large K) ----------------
        static_assert(!COOP || PPT == 1, "one pixel per thread");
        const unsigned full = live_mask;
        const int half = tid & 1;                    // this thread takes channels half, half + 2, ...
        T* colp = tile + (px0 & ~1);                 // the pair's first pixel
        // pass 1: packed max / arg-max over my channels, then merged with the partner's (ties -> lowest channel)
        // (channel rows are walked with running pointers: two rows per step)
        const size_t step = 2 * (size_t)PITCH;
        const T* rp = colp + (size_t)half * PITCH;
        typename Raw<T>::Max mt = Raw<T>::init(Raw<T>::ld(rp));
        Raw<T>::set_first(mt, half);
        rp += step;
#pragma unroll 4
        for (int c = half + 2; c < K; c += 2, rp += step) Raw<T>::update(mt, Raw<T>::ld(rp), c);
        float m0, m1;
        int a0, a1;
        Raw<T>::finish(mt, m0, m1, a0, a1);
        {
          const float pm0 = __shfl_xor_sync(full, m0, 1), pm1 = __shfl_xor_sync(full, m1, 1);
          const int pa0 = __shfl_xor_sync(full, a0, 1), pa1 = __shfl_xor_sync(full, a1, 1);
          if (pm0 > m0 || (pm0 == m0 && pa0 < a0)) { m0 = pm0; a0 = pa0; }
          if (pm1 > m1 || (pm1 == m1 && pa1 < a1)) { m1 = pm1; a1 = pa1; }
        }
        // pass 2: exponent sums of both pixels as packed pairs; old and new classes in separate loops
        const F2 nm2 = f2(-m0 * kLog2e, -m1 * kLog2e), l2e2 = f2b(kLog2e);
        auto exp_at = [&](const T* q) {
          float v0, v1;
          Raw<T>::unpack(Raw<T>::ld(q), v0, v1);
          const F2 arg = fma2(f2(v0, v1), l2e2, nm2);
          return f2(ex2_fast(f2lo(arg)), ex2_fast(f2hi(arg)));
        };
        const int new0 = max(old_cl, 1) + ((max(old_cl, 1) ^ half) & 1);  // my first new-class channel (never 0)
        // (channel 0 stays out of the loops: the foreground sum S_fg is accumulated directly, S - e_0 would cancel
        // when the background dominates)
        F2 so2 = f2b(0.f), sn2 = f2b(0.f);
        rp = colp + (size_t)(half == 0 ? 2 : 1) * PITCH;
#pragma unroll 4
        for (int c = (half == 0 ? 2 : 1); c < old_cl; c += 2, rp += step) so2 = add2(so2, exp_at(rp));
        rp = colp + (size_t)new0 * PITCH;
#pragma unroll 4
        for (int c = new0; c < K; c += 2, rp += step) sn2 = add2(sn2, exp_at(rp));
        {
          F2 po, pn;
          po.v = __shfl_xor_sync(full, so2.v, 1);
          pn.v = __shfl_xor_sync(full, sn2.v, 1);
          so2 = add2(so2, po);
          sn2 = add2(sn2, pn);
        }
        const F2 e02 = exp_at(colp);
        const F2 sf2 = add2(so2, sn2);  // foreground channels only
        const F2 sa2 = add2(sf2, e02);
        if (old_cl >= 1) so2 = add2(so2, e02);
        // per-pixel terms: thread `half` owns pixel `half` of the pair; coefficients are swapped by shuffle
        const float mx_me = half ? m1 : m0;
        amax[0] = half ? a1 : a0;
        pixel_terms(a, p.inv_n, s_norm, old_cl, y[0], is_ign[0], mx_me, half ? f2hi(sa2) : f2lo(sa2),
                    half ? f2hi(so2) : f2lo(so2), half ? f2hi(sf2) : f2lo(sf2), half ? f2hi(e02) : f2lo(e02), x0[0], xy[0],
                    seen[0], have_seen, zfoc[0], acc, pc[0], gfoc[0], dmask[0]);
        if (a.dlogits) {
          PixCoef po;
          po.cg0 = __shfl_xor_sync(full, pc[0].cg0, 1);
          po.cg1 = __shfl_xor_sync(full, pc[0].cg1, 1);
          po.cg2 = __shfl_xor_sync(full, pc[0].cg2, 1);
          po.d0 = __shfl_xor_sync(full, pc[0].d0, 1);
          const PixCoef& pa = half ? po : pc[0];   // pixel 0 of the pair
          const PixCoef& pb = half ? pc[0] : po;   // pixel 1 of the pair
          const F2 cgo = f2(pa.cg1, pb.cg1), cgn = f2(pa.cg2, pb.cg2);
          // pass 3: gradient rows of my channels, both pixels at once
          if (half == 0) {
            const F2 g = fma2(e02, f2(pa.cg0, pb.cg0), f2(-pa.d0, -pb.d0));
            Raw<T>::st(colp, f2lo(g), f2hi(g));
          }
          {
            const int c0 = half == 0 ? 2 : 1;
            T* wp = colp + (size_t)c0 * PITCH;
#pragma unroll 4
            for (int c = c0; c < old_cl; c += 2, wp += step) {
              const F2 g = mul2(exp_at(wp), cgo);
              Raw<T>::st(wp, f2lo(g), f2hi(g));
            }
            const int n1 = max(old_cl, 1) + ((max(old_cl, 1) ^ half) & 1);
            wp = colp + (size_t)n1 * PITCH;
#pragma unroll 4
            for (int c = n1; c < K; c += 2, wp += step) {
              const F2 g = mul2(exp_at(wp), cgn);
              Raw<T>::st(wp, f2lo(g), f2hi(g));
            }
          }
          __syncwarp(full);  // the partner's packed row stores are done before single elements are patched
          // the label's own channel, recomputed in fp32 so -dy is applied before rounding
          if (y[0] >= 0 && pc[0].dy != 0.f) {
            const int kk = y[0];
            const float cgk = kk == 0 ? pc[0].cg0 : (kk < old_cl ? pc[0].cg1 : pc[0].cg2);
            const float ey = ex2_fast(fmaf(xy[0], kLog2e, -mx_me * kLog2e));
            col[(size_t)kk * PITCH] = DT<T>::from_f(ey * cgk - pc[0].dy - (kk == 0 ? pc[0].d0 : 0.f));
          }
        }
      } else {
        // ---------------- generic path: three passes over the shared-memory tile ----------------
        float mx[PPT], nm[PPT], s_all[PPT], s_old[PPT], s_fg[PPT], e0[PPT], v[PPT];
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          mx[j] = -INFINITY;
          s_fg[j] = s_old[j] = 0.f;
        }
        #pragma unroll 8
        for (int c = 0; c < K; ++c) {
          Vec<T, PPT>::ld(col + (size_t)c * PITCH, v);
#pragma unroll
          for (int j = 0; j < PPT; ++j)
            if (v[j] > mx[j]) {
              mx[j] = v[j];
              amax[j] = c;
            }
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) nm[j] = -mx[j] * kLog2e;
        // channel 0 stays out of the loops: the foreground sum is accumulated directly (S - e_0 would cancel when
        // the background dominates)
        #pragma unroll 8
        for (int c = 1; c < old_cl; ++c) {
          Vec<T, PPT>::ld(col + (size_t)c * PITCH, v);
#pragma unroll
          for (int j = 0; j < PPT; ++j) s_old[j] += ex2_fast(fmaf(v[j], kLog2e, nm[j]));
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) s_fg[j] = s_old[j];
        #pragma unroll 8
        for (int c = max(old_cl, 1); c < K; ++c) {
          Vec<T, PPT>::ld(col + (size_t)c * PITCH, v);
#pragma unroll
          for (int j = 0; j < PPT; ++j) s_fg[j] += ex2_fast(fmaf(v[j], kLog2e, nm[j]));
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          e0[j] = ex2_fast(fmaf(x0[j], kLog2e, nm[j]));
          s_all[j] = s_fg[j] + e0[j];
          if (old_cl >= 1) s_old[j] += e0[j];
          pixel_terms(a, p.inv_n, s_norm, old_cl, y[j], is_ign[j], mx[j], s_all[j], s_old[j], s_fg[j], e0[j], x0[j],
                      xy[j], seen[j], have_seen, zfoc[j], acc, pc[j], gfoc[j], dmask[j]);
        }
        if (a.dlogits) {
          float g[PPT];
#pragma unroll
          for (int j = 0; j < PPT; ++j) g[j] = e0[j] * pc[j].cg0 - pc[j].d0;
          Vec<T, PPT>::st(col, g);
          #pragma unroll 8
          for (int c = 1; c < old_cl; ++c) {
            Vec<T, PPT>::ld(col + (size_t)c * PITCH, v);
#pragma unroll
            for (int j = 0; j < PPT; ++j) g[j] = ex2_fast(fmaf(v[j], kLog2e, nm[j])) * pc[j].cg1;
            Vec<T, PPT>::st(col + (size_t)c * PITCH, g);
          }
          #pragma unroll 8
          for (int c = max(old_cl, 1); c < K; ++c) {
            Vec<T, PPT>::ld(col + (size_t)c * PITCH, v);
#pragma unroll
            for (int j = 0; j < PPT; ++j) g[j] = ex2_fast(fmaf(v[j], kLog2e, nm[j])) * pc[j].cg2;
            Vec<T, PPT>::st(col + (size_t)c * PITCH, g);
          }
          // the label's own channel, recomputed in fp32 so -dy is applied before rounding
#pragma unroll
          for (int j = 0; j < PPT; ++j) {
            if (y[j] >= 0 && pc[j].dy != 0.f) {
              const int kk = y[j];
              const float cgk = kk == 0 ? pc[j].cg0 : (kk < old_cl ? pc[j].cg1 : pc[j].cg2);
              const float ey = ex2_fast(fmaf(xy[j], kLog2e, nm[j]));
              col[(size_t)kk * PITCH + j] = DT<T>::from_f(ey * cgk - pc[j].dy - (kk == 0 ? pc[j].d0 : 0.f));
            }
          }
        }
      }
    }
    // hand the stage back to the producer (gradient rows are complete)
    fence_proxy_async();
    mbar_arrive(&bar_done[s]);

    // ---- arg-max / mask stores -------------------------------------------------------------
    if (live) {
      if (a.preds) {
        int64_t* out = a.preds + (int64_t)b * HW + p0 + px0;
        if (PPT == 2 && px0 + 1 < npx && ((reinterpret_cast<uintptr_t>(out) & 15) == 0)) {
          *reinterpret_cast<longlong2*>(out) = make_longlong2((long long)amax[0], (long long)amax[PPT - 1]);
        } else {
#pragma unroll
          for (int j = 0; j < PPT; ++j)
            if (px0 + j < npx) out[j] = amax[j];
        }
      }
      if (a.distill_mask) {
        uint8_t* out = a.distill_mask + (int64_t)b * HW + p0 + px0;
        if (PPT == 2 && px0 + 1 < npx) {
          *reinterpret_cast<uchar2*>(out) = make_uchar2(dmask[0], dmask[PPT - 1]);
        } else {
#pragma unroll
          for (int j = 0; j < PPT; ++j)
            if (px0 + j < npx) out[j] = dmask[j];
        }
      }
    }

    // ---- focal gradient: adjoint of the bilinear up-sample ----------------------------------
    if (a.gz) {
      const unsigned full = 0xffffffffu;
      if (ROWTILE) {
        // all pixels share the row weights; reduce (g*(1-wx), g*wx) per low-res column.
        // A thread's PPT pixels are adjacent: combine them when they share the column.
        float c0 = gfoc[0] * (1.f - wx1[0]), c1 = gfoc[0] * wx1[0];
        const int key = cx0[0] * 2 + cdx[0];
        float d0 = 0.f, d1 = 0.f;
        int x2 = -1, dx2 = 0;
        if (PPT == 2) {
          const float f0 = gfoc[PPT - 1] * (1.f - wx1[PPT - 1]), f1 = gfoc[PPT - 1] * wx1[PPT - 1];
          const int k2 = cx0[PPT - 1] * 2 + cdx[PPT - 1];
          if (k2 == key) {
            c0 += f0;
            c1 += f1;
          } else {  // column boundary inside the pair: flushed on its own
            d0 = f0; d1 = f1; x2 = cx0[PPT - 1]; dx2 = cdx[PPT - 1];
          }
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float n0 = __shfl_down_sync(full, c0, o), n1 = __shfl_down_sync(full, c1, o);
          const int nk = __shfl_down_sync(full, key, o);
          if (lane + o < 32 && nk == key) {
            c0 += n0;
            c1 += n1;
          }
        }
        const int pk = __shfl_up_sync(full, key, 1);
        if (((lane == 0) || (pk != key)) && cx0[0] >= 0) {
          if (c0 != 0.f) atomicAdd(&gacc[cx0[0]], c0);
          if (c1 != 0.f) atomicAdd(&gacc[cx0[0] + cdx[0]], c1);
        }
        if (x2 >= 0) {
          if (d0 != 0.f) atomicAdd(&gacc[x2], d0);
          if (d1 != 0.f) atomicAdd(&gacc[x2 + dx2], d1);
        }
        consumer_sync();
        float* g = a.gz + (int64_t)b * a.h * a.w;
        const float wy0 = 1.f - ly_row.w1;
        for (int i = tid; i < a.w; i += kConsumers) {
          const float v = gacc[i];
          if (v != 0.f) {
            atomicAdd(g + ly_row.i0 * a.w + i, wy0 * v);
            if (ly_row.w1 != 0.f) atomicAdd(g + ly_row.i1 * a.w + i, ly_row.w1 * v);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          float c00 = gfoc[j] * (1.f - wy1g[j]) * (1.f - wx1[j]);
          float c01 = gfoc[j] * (1.f - wy1g[j]) * wx1[j];
          float c10 = gfoc[j] * wy1g[j] * (1.f - wx1[j]);
          float c11 = gfoc[j] * wy1g[j] * wx1[j];
          const int key = cell[j] * 4 + cdx[j] + 2 * (cell_dy[j] != 0);
          const int run_end = run_end_lane(key, lane);
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const float n00 = __shfl_down_sync(full, c00, o), n01 = __shfl_down_sync(full, c01, o);
            const float n10 = __shfl_down_sync(full, c10, o), n11 = __shfl_down_sync(full, c11, o);
            if (lane + o <= run_end) {
              c00 += n00; c01 += n01; c10 += n10; c11 += n11;
            }
          }
          const int pk = __shfl_up_sync(full, key, 1);
          if (((lane == 0) || (pk != key)) && cell[j] >= 0) {
            float* g = a.gz + (int64_t)b * a.h * a.w + cell[j];
            if (c00 != 0.f) atomicAdd(g, c00);
            if (c01 != 0.f) atomicAdd(g + cdx[j], c01);
            if (c10 != 0.f) atomicAdd(g + cell_dy[j], c10);
            if (c11 != 0.f) atomicAdd(g + cell_dy[j] + cdx[j], c11);
          }
        }
      }
    }

    // SCORE mode needs per-image sums: flush the accumulators per tile
    if (a.mode == BACS_PIX_SCORE) {
#pragma unroll
      for (int i = 0; i < BACS_NACC; ++i) {
        const float r = warp_sum(acc[i]);
        if (lane == 0) red_scratch[wid][i] = r;
        acc[i] = 0.f;
      }
      consumer_sync();
      if (tid < BACS_NACC) {
        float r = 0.f;
        for (int wv = 0; wv < kConsumerWarps; ++wv) r += red_scratch[wv][tid];
        const int tile_id = (int)blockIdx.x + k * (int)gridDim.x;
        p.partials[(int64_t)tile_id * BACS_NACC + tid] = (double)r;
      }
      consumer_sync();
    }
  }

  // ---- per-CTA partial sums ------------------------------------------------------------------
  if (a.mode != BACS_PIX_SCORE) {
#pragma unroll
    for (int i = 0; i < BACS_NACC; ++i) {
      const float r = warp_sum(acc[i]);
      if (lane == 0) red_scratch[wid][i] = r;
    }
    consumer_sync();
    if (tid < BACS_NACC) {
      double r = 0.0;
      for (int wv = 0; wv < kConsumerWarps; ++wv) r += (double)red_scratch[wv][tid];
      p.partials[(int64_t)blockIdx.x * BACS_NACC + tid] = r;
    }
  }
}

// Deterministic reduction of the partials: block 0 -> acc; in SCORE mode block 1+b -> score[b].
struct PixelEpilogue {
  const int32_t* ready;
  float* focal_scale_out;
  float* loss_out;
  float focal_weight, loss_coef;
  int loss_over_wsum;
};
__global__ void __launch_bounds__(256) pixel_reduce_kernel(const double* __restrict__ partials, int n_part,
                                                           int tiles_per_image, double* __restrict__ acc,
                                                           double* __restrict__ score, double inv_hw,
                                                           const PixelEpilogue ep) {
  __shared__ double scratch[8][BACS_NACC];
  __shared__ double total[BACS_NACC];
  const bool whole = blockIdx.x == 0;
  const int t0 = whole ? 0 : (blockIdx.x - 1) * tiles_per_image;
  const int t1 = whole ? n_part : t0 + tiles_per_image;
  // thread (g, i): accumulator i of partial rows g, g+32, ... (a partial row is 64 contiguous bytes)
  const int i = threadIdx.x & 7, g = threadIdx.x >> 3;
  double s = 0.0;
  pdl_wait();
  pdl_trigger();
  // eight partial rows in flight per thread (one row at a time is a chain of dependent L2 round trips: 6.7 us for the
  // 296 rows of a training step in the ncu launch list); same summation order
  for (int t = t0 + g; t < t1; t += 32 * 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int tt = t + 32 * u;
      v[u] = tt < t1 ? partials[(int64_t)tt * BACS_NACC + i] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) s += v[u];
  }
  s += __shfl_xor_sync(0xffffffffu, s, 8);
  s += __shfl_xor_sync(0xffffffffu, s, 16);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane < 8) scratch[wid][lane] = s;
  __syncthreads();
  if (threadIdx.x < BACS_NACC) {
    double r = 0.0;
    for (int wv = 0; wv < 8; ++wv) r += scratch[wv][threadIdx.x];
    if (whole) {
      acc[threadIdx.x] = r;
      total[threadIdx.x] = r;
    } else if (threadIdx.x == BACS_ACC_LOSS) {
      score[blockIdx.x - 1] = -r * inv_hw;
    }
  }
  if (!whole || (ep.focal_scale_out == nullptr && ep.loss_out == nullptr)) return;
  __syncthreads();
  if (threadIdx.x == 0) {  // the step's scalar epilogue (focal normaliser, loss value)
    const double kept = total[BACS_ACC_KEPT];
    const bool on = (ep.ready == nullptr || *ep.ready != 0) && total[BACS_ACC_BG] > 0.0 && kept > 0.0;
    const double fs = on ? (double)ep.focal_weight / kept : 0.0;
    if (ep.focal_scale_out) *ep.focal_scale_out = (float)fs;
    if (ep.loss_out) {
      double main = (double)ep.loss_coef * total[BACS_ACC_LOSS];
      if (ep.loss_over_wsum) main /= total[BACS_ACC_WSUM];
      *ep.loss_out = (float)(main + fs * total[BACS_ACC_FOCAL]);
    }
  }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
    (void)cudaGetLastError();
  }
  return fn;
}

// [B,K,H,W] as the 3-D tensor (H*W, K, B) with boxes of 256 pixels x K channels x 1 image
static bool make_tile_map(CUtensorMap* map, const void* base, int dtype, int B, int K, int64_t HW, unsigned box_px = 256u) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || K > 256) return false;
  const size_t es = dtype_size(dtype);
  const CUtensorMapDataType dt = dtype == BACS_F32    ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : dtype == BACS_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                      : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)K, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)HW * es, (cuuint64_t)HW * K * es};
  const cuuint32_t box[3] = {box_px, (cuuint32_t)K, 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return fn(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// seen logits [B,T,h,w] as the 4-D tensor (w, h, T, B); one box = rows (i0, i0+1) of every head
static bool make_z_map(CUtensorMap* map, const float* z, int B, int T, int h, int w) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || w > 256 || T > 256 || (w * 4) % 16 != 0 || (reinterpret_cast<uintptr_t>(z) & 15) != 0) return false;
  const cuuint64_t dims[4] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t strides[3] = {(cuuint64_t)w * 4, (cuuint64_t)h * w * 4, (cuuint64_t)T * h * w * 4};
  const cuuint32_t box[4] = {(cuuint32_t)w, 2u, (cuuint32_t)T, 1u};
  const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(z), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Plan of the shared-memory tile kernels.  Returns the variant: 2 the training-step kernel, 1 the K <= 24 register
// kernel, 0 the generic tile kernel, -1 when K fits no shared-memory tile.
static int make_plan(const bacs_pixel_args& a, PixelPlan* plan) {
  const size_t es = dtype_size(a.dtype);
  const int64_t HW = (int64_t)a.H * a.W;
  const int sms = sm_count();
  const size_t extra = (a.z ? (size_t)a.T * a.w * 4 : 0) + (size_t)(a.w + 1) * 4 + 64;
  const size_t cap = 220 * 1024;
  auto aligned16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };

  // ---- fast path: K <= 24 logits per pixel stay in registers, full 512-pixel tiles, TMA ring ----
  const bool fast_ok = a.K <= 24 && HW % 512 == 0 && (HW * es) % 16 == 0 && aligned16(a.logits) &&
                       aligned16(a.labels) && (!a.dlogits || aligned16(a.dlogits)) && (!a.preds || aligned16(a.preds)) &&
                       (!a.distill_mask || (reinterpret_cast<uintptr_t>(a.distill_mask) & 1) == 0);
  if (fast_ok) {
    static const int kregs[7] = {4, 8, 12, 16, 20, 21, 24};
    int kreg = 24;
    for (int i = 0; i < 7; ++i)
      if (kregs[i] >= a.K) {
        kreg = kregs[i];
        break;
      }
    // 4 stages of {kreg logit rows, 512 int64 labels, seen-head rows} + one [T][8] float2 strip per warp
    const size_t zrows = a.z ? (((size_t)a.T * 2 * a.w * 4 + 127) & ~(size_t)127) : 0;
    const size_t stage = (size_t)kreg * 512 * es + 4096 + zrows;
    const size_t tail = (a.z ? (size_t)8 * a.T * 8 * 8 : 0) + 64;
    // row tiles: a tile lies inside one image row and 64 pixels touch <= 6 low-res columns
    const bool rowtile = a.z != nullptr && a.W % 512 == 0 && a.seen_scale >= 16 && a.w % 4 == 0 &&
                         (reinterpret_cast<uintptr_t>(a.z) & 15) == 0;
    // 228 KB of shared memory per SM, 1 KB reserved per resident CTA, < 0.5 KB static
    auto two_fit = [](size_t smem) { return 2 * (smem + 1024 + 512) <= (size_t)228 * 1024; };
    // the training-step kernel (needs the tensor maps); it also runs with a 3-stage ring when that is what lets two
    // CTAs share an SM
    const bool wce = rowtile && a.mode == BACS_PIX_WEIGHTED_CE && !a.seen_max && encode_tiled_fn() != nullptr &&
                     a.w <= 256 && a.T <= 256 && a.K <= 256;
    int stages = 4;
    if (wce && !two_fit(4 * stage + tail) && two_fit(3 * stage + tail)) stages = 3;
    const size_t smem = (size_t)stages * stage + tail;
    if (smem + 1024 <= cap) {
      const int per_sm = two_fit(smem) ? 2 : 1;
      const int64_t tiles = HW / 512 * a.B;
      plan->coop = 0;
      plan->ppt = 2;
      plan->P = 512;
      plan->kreg = kreg;
      plan->stages = stages;
      plan->smem = smem;
      plan->grid = (int)std::min<int64_t>(tiles, (int64_t)sms * per_sm);
      plan->rowtile = rowtile ? 1 : 0;
      return wce ? 2 : 1;
    }
  }

  // ---- generic path: any K that fits a shared-memory tile, ragged / unaligned shapes ----
  plan->kreg = 0;
  for (int min_stages = 2; min_stages >= 1; --min_stages)
    for (int ppt = 2; ppt >= 1; --ppt) {
      if (ppt == 2 && (HW & 1)) continue;  // pixel pairs need even image sizes
      const int P = ppt * kConsumers;
      // one pixel per thread and even images: lane pairs walk the channels together on padded rows (see the kernel)
      const bool coop = ppt == 1 && (HW & 1) == 0 && a.K >= 2;
      const size_t tile = (size_t)a.K * ((size_t)P * es + (coop ? 64 : 0));
      int stages = 0;
      for (int st = 3; st >= min_stages; --st)
        if ((size_t)st * tile + extra + 1024 <= cap) {
          stages = st;
          break;
        }
      if (!stages) continue;
      const int64_t tiles = (HW + P - 1) / P * a.B;
      size_t smem = (size_t)stages * tile + extra;
      int per_sm = 1;
      if (ppt == 1) {  // (measured at K = 151: 2 CTAs x 1 stage 1.57 ms, 1 CTA x 2 stages 1.75 ms)
        // large K: one pixel per thread.  Two CTAs per SM double the warps that hide latency; when two stages each
        // do not fit, one stage each still overlaps -- one CTA computes while the other one loads / stores.
        auto two_fit = [](size_t sm) { return 2 * (sm + 1024 + 512) <= (size_t)228 * 1024; };
        for (int st = std::min(stages, 2); st >= 1; --st)
          if (two_fit((size_t)st * tile + extra)) {
            stages = st;
            smem = (size_t)st * tile + extra;
            per_sm = 2;
            break;
          }
      }
      plan->ppt = ppt;
      plan->coop = coop ? 1 : 0;
      plan->P = P;
      plan->stages = stages;
      plan->smem = smem;
      plan->grid = (int)std::min<int64_t>(tiles, (int64_t)sms * per_sm);
      plan->rowtile = (a.z != nullptr && P <= a.W && a.W % P == 0) ? 1 : 0;
      return 0;
    }
  return -1;
}

}  // namespace bacs

#include "pixel_lowres.cuh"  // the same loss evaluated from low-res logits (up-sample + adjoint fused)
#include "pixel_stream.cuh"  // large class counts: two streaming passes instead of shared-memory tiles
#include "pixel_regs.cuh"    // large class counts in 16-bit storage: one pass, the channel column in registers

namespace bacs {

struct StreamPlan {
  int blocks_x;
  size_t part_bytes, coef_bytes;
};

// K >= 64 on 16-byte aligned, vector-divisible images (everything else stays on the tile kernel)
static bool make_stream_plan(const bacs_pixel_args& a, StreamPlan* plan) {
  const int64_t HW = (int64_t)a.H * a.W;
  const int n = a.dtype == BACS_F32 ? 4 : 8;
  auto al = [](const void* p, uintptr_t m) { return (reinterpret_cast<uintptr_t>(p) & (m - 1)) == 0; };
  if (a.K < 64 || HW % n != 0 || !al(a.logits, 16) || !al(a.labels, 16)) return false;
  if (a.dlogits && !al(a.dlogits, 16)) return false;
  if (a.preds && !al(a.preds, 16)) return false;
  if (a.distill_mask && !al(a.distill_mask, 4)) return false;
  const int64_t groups = HW / n;
  int64_t bx = (groups + kStreamThreads - 1) / kStreamThreads;
  const int64_t cap = std::max<int64_t>(1, (int64_t)sm_count() * 4);  // per image
  if (bx > cap) bx = cap;
  plan->blocks_x = (int)bx;
  plan->part_bytes = align_up((size_t)bx * a.B * BACS_NACC * sizeof(double), 256);
  plan->coef_bytes = a.dlogits ? align_up((size_t)6 * HW * a.B * sizeof(float), 256) : 0;
  return true;
}

// 16-bit logits with 64 <= K <= kRegsKMax on images of a multiple of 256 pixels: one pass with the channel column of a
// pixel pair in the registers of two lanes (pixel_regs.cuh).  BACS_NO_REGS=1 leaves these shapes to the streaming
// passes (the reference the register-column kernel is tested against).
static bool make_regs_plan(const bacs_pixel_args& a, StreamPlan* plan) {
  if (getenv("BACS_NO_REGS")) return false;
  const int64_t HW = (int64_t)a.H * a.W;
  auto al = [](const void* p, uintptr_t m) { return (reinterpret_cast<uintptr_t>(p) & (m - 1)) == 0; };
  if (a.dtype == BACS_F32 || a.K < 64 || a.K > kRegsKMax || HW % 256 != 0 || encode_tiled_fn() == nullptr) return false;
  if (a.mode == BACS_PIX_SCORE) return false;  // (per-image sums: streaming path)
  if (!al(a.logits, 16) || !al(a.labels, 8) || (a.dlogits && !al(a.dlogits, 4))) return false;
  const int64_t tiles = HW / kRegsNT * a.B;
  if (tiles > 0x3fffffff) return false;
  plan->blocks_x = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * kRegsCTAs);  // persistent: one wave
  plan->part_bytes = align_up((size_t)plan->blocks_x * BACS_NACC * sizeof(double), 256);
  plan->coef_bytes = 0;
  return true;
}

struct LowresPlan {
  int SX, R, groups, nsrc_max, grid;
  bool exact;  // W == SX * lw: the instantiation with compile-time pixel offsets
  size_t smem, part_bytes, g32_bytes;
};

// host copy of lerp_half_pixel's source coordinate (fp32, op by op)
static float host_src(int dst, float scale) {
  volatile float t = (float)dst + 0.5f;
  volatile float m = scale * t;
  float src = m - 0.5f;
  return src < 0.f ? 0.f : src;
}

// host copy of lerp_half_pixel
static void host_half_pixel(int dst, int in_size, float scale, int* i0, int* i1) {
  *i0 = std::min((int)host_src(dst, scale), in_size - 1);
  *i1 = *i0 + (*i0 < in_size - 1 ? 1 : 0);
}

// host copy of lowres_span_start (pixel_lowres.cuh)
static int host_span_start(int j, int lw, int W, float scale) {
  auto owner = [&](int x) {
    volatile float h = host_src(x, scale) + 0.5f;
    return (int)h;
  };
  if (j >= lw) return W;
  int x = (int)((int64_t)j * W / lw);
  while (x > 0 && owner(x - 1) >= j) --x;
  while (x < W && owner(x) < j) ++x;
  return x;
}

// Accepted geometry: W == SX * lw with SX 8 or 16 and H a multiple of lh, or the network's output stride s = 16 or 8
// applied to any input, lh == ceil(H / s) and lw == ceil(W / s) (DeepLab's padded stride-2 convolutions; s = 16 where
// both match).  The seen heads (a.z) need the first form.
static bool make_lowres_plan(const bacs_pixel_args& a, int lh, int lw, LowresPlan* plan) {
  if (lh <= 0 || lw <= 0 || lw > kLowresThreads || a.K > 255) return false;
  int SX = 0;
  bool exact = false;
  if (a.W % lw == 0 && a.H % lh == 0 && (a.W / lw == 16 || a.W / lw == 8)) {
    SX = a.W / lw;
    exact = true;
  } else {
    for (int s : {16, 8})
      if (lh == (a.H + s - 1) / s && lw == (a.W + s - 1) / s) {
        SX = s;
        break;
      }
    if (SX == 0 || a.z) return false;
    exact = a.W == SX * lw;  // whole spans in x; the kernel's rows take any H
    if (!exact) {            // every column's span fits the kernel's SX-pixel arrays
      const float hx = hp_scale(lw, a.W);
      for (int j = 0, x0 = 0; j < lw; ++j) {
        const int x1 = host_span_start(j + 1, lw, a.W, hx);
        if (x1 - x0 > SX) return false;
        x0 = x1;
      }
    }
  }
  int R = 1;
  while (2 * R * lw <= kLowresThreads && 2 * R <= a.H) R *= 2;
  const float hy = hp_scale(lh, a.H);
  int groups, nsrc;
  size_t smem;
  for (;; R /= 2) {  // a row group may touch at most kLowresMaxSrc source rows, and its staging must fit
    groups = (a.H + R - 1) / R;
    nsrc = 1;
    for (int g = 0; g < groups; ++g) {
      int f0, f1, l0, l1;
      host_half_pixel(g * R, lh, hy, &f0, &f1);
      host_half_pixel(std::min(g * R + R, a.H) - 1, lh, hy, &l0, &l1);
      nsrc = std::max(nsrc, l1 - f0 + 1);
    }
    smem = ((size_t)nsrc * a.K * (lw + 2) + (size_t)3 * R * kLowresChunk * lw + (size_t)nsrc * R +
            (a.z ? (size_t)R * a.T * a.w : 0) + (size_t)R * (a.w + 1)) * 4 + 16;
    if ((nsrc <= kLowresMaxSrc && smem <= kLowresMaxSmem) || R == 1) break;
  }
  plan->SX = SX;
  plan->exact = exact;
  plan->R = R;
  plan->groups = groups;
  plan->nsrc_max = nsrc;
  plan->grid = groups * a.B;
  plan->smem = smem;
  plan->part_bytes = align_up((size_t)plan->grid * BACS_NACC * sizeof(double), 256);
  plan->g32_bytes = (a.dlogits && a.dtype != BACS_F32) ? align_up((size_t)a.B * a.K * lh * lw * 4, 256) : 0;
  return plan->smem <= kLowresMaxSmem;
}

// What bacs_pixel_loss runs for `a`.  The kernel is chosen here alone, so that bacs_pixel_kernel_variant and
// bacs_pixel_workspace_bytes report what runs.
struct PixelRoute {
  int variant;       // 0 generic tiles, 1 K <= 24 registers, 2 training step (plan); 4 streaming passes, 5 register
                     // column (sp); -1 when K fits no shared-memory tile
  PixelPlan plan;
  StreamPlan sp;
  int64_t n_part, part_per_image;  // partial rows of pixel_reduce_kernel; per image in SCORE mode
  size_t workspace;  // bacs_pixel_workspace_bytes
};

static PixelRoute pixel_route(const bacs_pixel_args& a) {
  PixelRoute r = {};
  if (make_regs_plan(a, &r.sp)) {
    r.variant = 5;
    r.n_part = r.part_per_image = r.sp.blocks_x;
  } else if (make_stream_plan(a, &r.sp)) {
    r.variant = 4;
    r.n_part = (int64_t)r.sp.blocks_x * a.B;
    r.part_per_image = r.sp.blocks_x;
  } else {
    r.variant = make_plan(a, &r.plan);
    if (r.variant < 0) return r;
    r.part_per_image = ((int64_t)a.H * a.W + r.plan.P - 1) / r.plan.P;  // tiles per image
    r.n_part = a.mode == BACS_PIX_SCORE ? r.part_per_image * a.B : r.plan.grid;
    r.workspace = align_up((size_t)r.n_part * BACS_NACC * sizeof(double), 256);
    return r;
  }
  r.workspace = r.sp.part_bytes + r.sp.coef_bytes;
  return r;
}

// The argument checks of bacs_pixel_loss and bacs_pixel_loss_lowres; `fn` starts each message.
static int check_pixel_args(const bacs_pixel_args* a, const char* fn) {
  BACS_REQUIRE(a && a->logits && a->labels && a->acc, "%s: logits, labels and acc are required", fn);
  BACS_REQUIRE(a->B > 0 && a->K > 0 && a->H > 0 && a->W > 0, "%s: bad shape", fn);
  BACS_REQUIRE(a->ignore_index >= a->K || a->ignore_index < 0, "%s: ignore_index inside the class range", fn);
  BACS_REQUIRE(a->mode >= 0 && a->mode <= BACS_PIX_SCORE, "%s: unknown mode %d", fn, a->mode);
  BACS_REQUIRE(a->dtype >= 0 && a->dtype <= BACS_F16, "%s: unknown dtype %d", fn, a->dtype);
  if (a->z) {
    BACS_REQUIRE(a->T > 0 && a->h > 0 && a->w > 0, "%s: seen logits given without T/h/w", fn);
    BACS_REQUIRE(a->seen_scale > 0 && a->H == a->h * a->seen_scale && a->W == a->w * a->seen_scale,
                 "%s: H,W must equal h,w * seen_scale (the reference's nn.Upsample(scale_factor))", fn);
  }
  if (a->gz) BACS_REQUIRE(a->z && a->focal_head >= 0 && a->focal_head < a->T, "%s: focal head out of range", fn);
  if (a->mode == BACS_PIX_WEIGHTED_CE)
    BACS_REQUIRE(a->old_cl >= 1 && (a->z || a->seen_max),
                 "%s: WEIGHTED_CE needs old_cl >= 1 and the seen logits / probabilities", fn);
  if (a->mode != BACS_PIX_WEIGHTED_CE && a->dlogits)
    BACS_REQUIRE(a->hist, "%s: CE-type gradients need the label histogram", fn);
  if (a->mode == BACS_PIX_SCORE)
    BACS_REQUIRE(a->score && !a->dlogits, "%s: SCORE mode needs score and no gradient", fn);
  return BACS_OK;
}

// pixel_reduce_kernel over the n_part partial rows (per_image of them per image in SCORE mode), with the step's
// scalar epilogue
static void launch_pixel_reduce(const bacs_pixel_args& a, const double* partials, int n_part, int per_image,
                                cudaStream_t s) {
  const PixelEpilogue ep = {a.ready, a.focal_scale_out, a.loss_out, a.focal_weight, a.loss_coef, a.loss_over_wsum};
  launch_pdl(pixel_reduce_kernel, dim3(1 + (a.mode == BACS_PIX_SCORE ? a.B : 0)), dim3(256), 0, s, partials, n_part,
             per_image, a.acc, a.score, 1.0 / ((double)a.H * (double)a.W), ep);
}

template <typename T>
static int launch_tile_kernel(const PixelParams& p, const PixelPlan& plan, cudaStream_t s) {
  auto kern = plan.ppt == 2 ? (plan.rowtile ? pixel_loss_kernel<T, 2, true> : pixel_loss_kernel<T, 2, false>)
              : plan.coop ? (plan.rowtile ? pixel_loss_kernel<T, 1, true, true> : pixel_loss_kernel<T, 1, false, true>)
                          : (plan.rowtile ? pixel_loss_kernel<T, 1, true> : pixel_loss_kernel<T, 1, false>);
  return launch_pixel_kernel("bacs_pixel_loss", false, kern, dim3(plan.grid), dim3(kConsumers + 32), plan.smem, s,
                             p);
}

}  // namespace bacs

using namespace bacs;

extern "C" {

size_t bacs_pixel_lowres_workspace_bytes(const bacs_pixel_args* a, int32_t lh, int32_t lw) {
  if (!a) return 0;
  LowresPlan plan;
  if (!make_lowres_plan(*a, lh, lw, &plan)) return 0;
  return plan.part_bytes + plan.g32_bytes;
}

int bacs_pixel_loss_lowres(const bacs_pixel_args* a, int32_t lh, int32_t lw, void* workspace, size_t workspace_bytes,
                           void* stream) {
  int rc = check_pixel_args(a, "bacs_pixel_loss_lowres");
  if (rc != BACS_OK) return rc;
  LowresPlan plan;
  if (!make_lowres_plan(*a, lh, lw, &plan)) {
    set_error("bacs_pixel_loss_lowres: unsupported geometry (H=%d W=%d lh=%d lw=%d K=%d%s): needs W == s*lw with "
              "s = 8 or 16 and H a multiple of lh, or lh == ceil(H/s) and lw == ceil(W/s) for s = 8 or 16 (not with "
              "the seen logits z); lw <= 256, K <= 255, staging within %zu bytes of shared memory",
              a->H, a->W, lh, lw, a->K, a->z ? ", seen logits z given" : "", kLowresMaxSmem);
    return BACS_ERR_UNSUPPORTED;
  }
  if (!workspace || workspace_bytes < plan.part_bytes + plan.g32_bytes) {
    set_error("bacs_pixel_loss_lowres: workspace too small (%zu bytes)", workspace_bytes);
    return BACS_ERR_WORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n_low = (int64_t)a->B * a->K * lh * lw;
  LowresParams p;
  p.a = *a;
  p.g32 = nullptr;
  if (a->dlogits) {
    p.g32 = a->dtype == BACS_F32 ? reinterpret_cast<float*>(a->dlogits)
                                 : reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(workspace) + plan.part_bytes);
    if (cudaMemsetAsync(p.g32, 0, (size_t)n_low * 4, s) != cudaSuccess) {
      set_error("bacs_pixel_loss_lowres: memset failed");
      return BACS_ERR_CUDA;
    }
  }
  p.lh = lh;
  p.lw = lw;
  p.R = plan.R;
  p.groups_per_image = plan.groups;
  p.nsrc_max = plan.nsrc_max;
  p.hy = hp_scale(lh, a->H);
  p.inv_n = (float)(1.0 / ((double)a->B * (double)a->H * (double)a->W));
  p.sy = a->z ? ac_scale(a->h, a->H) : 0.f;
  p.sx = a->z ? ac_scale(a->w, a->W) : 0.f;
  p.partials = reinterpret_cast<double*>(workspace);
  p.hx = hp_scale(lw, a->W);
  auto kern = plan.exact ? (plan.SX == 16 ? pixel_lowres_kernel<16, true> : pixel_lowres_kernel<8, true>)
                         : (plan.SX == 16 ? pixel_lowres_kernel<16, false> : pixel_lowres_kernel<8, false>);
  rc = launch_pixel_kernel("bacs_pixel_loss_lowres", false, kern, dim3(plan.grid), dim3(kLowresThreads), plan.smem, s,
                           p);
  if (rc != BACS_OK) return rc;
  BACS_CHECK_LAUNCH("bacs_pixel_loss_lowres");
  if (a->dlogits && a->dtype != BACS_F32) {
    const int nb = (int)((n_low + 255) / 256);
    if (a->dtype == BACS_BF16)
      lowres_cast_kernel<__nv_bfloat16><<<nb, 256, 0, s>>>(p.g32, reinterpret_cast<__nv_bfloat16*>(a->dlogits), n_low);
    else
      lowres_cast_kernel<__half><<<nb, 256, 0, s>>>(p.g32, reinterpret_cast<__half*>(a->dlogits), n_low);
    BACS_CHECK_LAUNCH("bacs_pixel_loss_lowres(cast)");
  }
  launch_pixel_reduce(*a, p.partials, plan.grid, plan.groups, s);
  BACS_CHECK_LAUNCH("bacs_pixel_loss_lowres(reduce)");
  return BACS_OK;
}

size_t bacs_pixel_workspace_bytes(const bacs_pixel_args* a) { return a ? pixel_route(*a).workspace : 0; }

int bacs_pixel_kernel_variant(const bacs_pixel_args* a) { return a ? pixel_route(*a).variant : -1; }

int bacs_pixel_loss(const bacs_pixel_args* a, void* workspace, size_t workspace_bytes, bacs_stream_t stream) {
  int rc = check_pixel_args(a, "bacs_pixel_loss");
  if (rc != BACS_OK) return rc;
  const PixelRoute r = pixel_route(*a);
  if (r.variant < 0) {
    set_error("bacs_pixel_loss: K=%d too large for a shared-memory tile", a->K);
    return BACS_ERR_UNSUPPORTED;
  }
  const bool tiles = r.variant <= 2;
  BACS_REQUIRE(!tiles || r.part_per_image * a->B < 0x7fffffff, "bacs_pixel_loss: too many tiles");
  // (the tile kernels write their partial rows alone; bacs_pixel_workspace_bytes rounds those up to 256 bytes)
  const size_t need = tiles ? (size_t)r.n_part * BACS_NACC * sizeof(double) : r.workspace;
  if (!workspace || workspace_bytes < need) {
    set_error("bacs_pixel_loss: workspace too small (%zu bytes)", workspace_bytes);
    return BACS_ERR_WORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  double* partials = reinterpret_cast<double*>(workspace);
  const int64_t HW = (int64_t)a->H * a->W;
  const float inv_n = (float)(1.0 / ((double)a->B * (double)HW));
  const float sy = a->z ? ac_scale(a->h, a->H) : 0.f, sx = a->z ? ac_scale(a->w, a->W) : 0.f;
  if (!tiles) {
    StreamParams q;
    q.a = *a;
    q.partials = partials;
    // the streaming passes' coefficient planes follow the partials; the register-column kernel only tests the pointer
    // (a gradient is wanted)
    q.coef = a->dlogits ? reinterpret_cast<float*>(ws + (r.variant == 4 ? r.sp.part_bytes : 0)) : nullptr;
    q.blocks_x = r.sp.blocks_x;
    q.b0 = 0;
    q.inv_n = inv_n;
    q.sy = sy;
    q.sx = sx;
    if (r.variant == 5) {  // large K, 16-bit logits: one pass, channel column in registers (pixel_regs.cuh)
      RegsParams rq;
      rq.s = q;
      rq.tiles_per_image = (int)(HW / kRegsNT);
      rq.n_tiles = rq.tiles_per_image * a->B;
      if (!make_tile_map(&rq.tmap_in, a->logits, a->dtype, a->B, a->K, HW, (unsigned)kRegsNT)) {
        set_error("bacs_pixel_loss: cuTensorMapEncodeTiled failed for the logits");
        return BACS_ERR_CUDA;
      }
      auto kern = a->dtype == BACS_BF16 ? pixel_regs_kernel<__nv_bfloat16, kRegsKH, kRegsNT, kRegsCTAs>
                                        : pixel_regs_kernel<__half, kRegsKH, kRegsNT, kRegsCTAs>;
      rc = launch_pixel_kernel("bacs_pixel_loss", false, kern, dim3(r.sp.blocks_x), dim3(kRegsNT),
                               (size_t)a->K * kRegsNT * 2 + 128, s, rq);
      if (rc != BACS_OK) return rc;
      BACS_CHECK_LAUNCH("bacs_pixel_loss(register column)");
    } else {  // large K: two streaming passes (pixel_stream.cuh)
      // (launching a few images at a time so that pass B re-reads them from the 126 MB L2 was measured: 1 / 2 / 4 / 8
      //  images per launch pair 2.67 / 1.69 / 1.66 / 1.48 ms against 1.33 ms for all 24 at once -- under-filled
      //  launches cost more than the second HBM read)
      const dim3 grid((unsigned)r.sp.blocks_x, (unsigned)a->B);
      BACS_DISPATCH_DTYPE(a->dtype, TT, { pixel_stream_stats_kernel<TT><<<grid, kStreamThreads, 0, s>>>(q); });
      BACS_CHECK_LAUNCH("bacs_pixel_loss(stream stats)");
      if (a->dlogits) {
        BACS_DISPATCH_DTYPE(a->dtype, TT, { pixel_stream_grad_kernel<TT><<<grid, kStreamThreads, 0, s>>>(q); });
        BACS_CHECK_LAUNCH("bacs_pixel_loss(stream grad)");
      }
    }
  } else {
    const size_t es = dtype_size(a->dtype);
    PixelParams p;
    p.a = *a;
    p.P = r.plan.P;
    p.tiles_per_image = (int)r.part_per_image;
    p.n_tiles = (int)(r.part_per_image * a->B);
    p.stages = r.plan.stages;
    p.inv_n = inv_n;
    p.sy = sy;
    p.sx = sx;
    p.partials = partials;
    p.use_tmap = 0;
    if (r.variant >= 1) {
      const bool ok_in = make_tile_map(&p.tmap_in, a->logits, a->dtype, a->B, a->K, HW);
      const bool ok_out = !a->dlogits || make_tile_map(&p.tmap_out, a->dlogits, a->dtype, a->B, a->K, HW);
      const bool ok_z = !(r.plan.rowtile && a->z) || make_z_map(&p.tmap_z, a->z, a->B, a->T, a->h, a->w);
      p.use_tmap = (ok_in && ok_out && ok_z) ? 1 : 0;
    }
    p.use_bulk = (((HW * es) % 16 == 0) && ((reinterpret_cast<uintptr_t>(a->logits) & 15) == 0) &&
                  (!a->dlogits || (reinterpret_cast<uintptr_t>(a->dlogits) & 15) == 0))
                     ? 1
                     : 0;
    // the training-step kernel needs the tensor maps: without them a 4-stage ring runs on pixel_fast_kernel, while a
    // 3-stage ring (planned for the training-step kernel alone) has no kernel to run on
    int variant = r.variant;
    if (variant == 2 && !p.use_tmap) {
      if (r.plan.stages != 4) {
        set_error("bacs_pixel_loss: tensor-map creation failed for the 3-stage training kernel");
        return BACS_ERR_CUDA;
      }
      variant = 1;
    }
    if (variant == 2) {
      switch (a->dtype) {
        case BACS_F32: rc = launch_pixel_wce_f32(p, r.plan, s); break;
        case BACS_BF16: rc = launch_pixel_wce_bf16(p, r.plan, s); break;
        default: rc = launch_pixel_wce_f16(p, r.plan, s); break;
      }
    } else if (variant == 1) {
      switch (a->dtype) {
        case BACS_F32: rc = launch_pixel_fast_f32(p, r.plan, s); break;
        case BACS_BF16: rc = launch_pixel_fast_bf16(p, r.plan, s); break;
        default: rc = launch_pixel_fast_f16(p, r.plan, s); break;
      }
    } else {
      BACS_DISPATCH_DTYPE(a->dtype, TT, { rc = launch_tile_kernel<TT>(p, r.plan, s); });
    }
    if (rc != BACS_OK) return rc;
    BACS_CHECK_LAUNCH("bacs_pixel_loss");
  }
  launch_pixel_reduce(*a, partials, (int)r.n_part, (int)r.part_per_image, s);
  BACS_CHECK_LAUNCH("bacs_pixel_loss(reduce)");
  return BACS_OK;
}

}  // extern "C"
