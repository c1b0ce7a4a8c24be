// The training-step specialisation of the fused per-pixel kernel: background-weighted unbiased CE
// (training/loss_utils.py:542-585) with the seen heads given at stride 16 (networks/bg_detector.py:13-15),
// optional seen-detector focal term (loss/base_loss.py:255-272), distill mask (loss/bacs_loss.py:282-285),
// arg-max (loss/bacs_loss.py:255) and d(loss)/d(logits), for K <= 24 and tiles that are whole 512-pixel
// pieces of one image row.
//
// Same data movement as pixel_fast_kernel (4-stage ring of 3-D tensor-map TMA tiles, one issuing lane,
// gradients leave through TMA stores) but the per-pixel instruction stream is cut to the bone:
//   * seen heads: the warp's y-interpolated strip is stored as (z[c], z[c+1]) pairs -> one LDS.64,
//     2 FMUL, 1 FADD, 1 FMNMX per head and pixel, no per-head selects;
//   * the three label cases of the CE are evaluated select-only (no divergent branches), with
//     lg2/rcp on S, S_old and S - e_0 only;
//   * gradient coefficients are chosen per group of four channels by uniform branches;
//   * padding channels (K < KREG) are predicated at the load, nothing is predicated at the store;
//   * the focal gradient (adjoint of the x16 up-sample) is reduced over groups of 8 lanes: 16 adjacent
//     pixels touch at most three low-res columns;
//   * pixel counters are 8-bit fields of one register.
#pragma once
#include "pixel_fast.cuh"

namespace bacs {

__device__ __forceinline__ void mbar_wait_sleepy(uint64_t* bar, uint32_t parity) {
  // try_wait with a suspend-time hint: a waiting warp parks in the barrier unit instead of spinning
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAITS_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra WAITS_DONE;\n"
      "bra WAITS_LOOP;\n"
      "WAITS_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(0x989680)
      : "memory");
}

__device__ __forceinline__ float lg2_fast(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

constexpr float kLn2 = 0.6931471805599453f;

// smallest K served by the kernel instantiated for KREG register rows
__host__ __device__ constexpr int wce_kmin(int kreg) {
  return kreg == 4 ? 1 : kreg == 8 ? 5 : kreg == 12 ? 9 : kreg == 16 ? 13 : kreg == 20 ? 17 : kreg == 21 ? 21 : 22;
}

template <typename T> struct NegInf;
template <> struct NegInf<float> {
  __device__ static __forceinline__ float2 pair() { return make_float2(-INFINITY, -INFINITY); }
};
template <> struct NegInf<__nv_bfloat16> {
  __device__ static __forceinline__ uint32_t pair() { return 0xff80ff80u; }
};
template <> struct NegInf<__half> {
  __device__ static __forceinline__ uint32_t pair() { return 0xfc00fc00u; }
};

// Shared memory (dynamic): 4 stages of { [2][KREG][256] logits, 512 int64 labels, [T][2][w] seen-head rows }
// followed by one warp-private [T][8] strip of float2 per warp.
// STD: the reference's hyper-parameters (gamma = focal gamma = 2, no alpha weighting, ukd) folded at compile time.
template <typename T, int KREG, bool STD, int S>
__global__ void __launch_bounds__(kFastThreads, 2) pixel_wce_kernel(const __grid_constant__ PixelParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t bar_full[4];
  __shared__ uint64_t bar_done[4];
  __shared__ float red_scratch[8][BACS_NACC];

  constexpr int P = kFastP;
  static_assert(S == 3 || S == 4, "ring depth");
  constexpr int KMIN = wce_kmin(KREG);
  constexpr size_t tile_bytes_smem = (size_t)KREG * P * sizeof(T);
  const bacs_pixel_args& a = p.a;
  const int K = a.K, TH = a.T;
  const int tid = threadIdx.x;
  const int lane = tid & 31, wid = tid >> 5;
  const int64_t HW = (int64_t)a.H * a.W;
  const uint32_t zrow_bytes = (uint32_t)(TH * 2 * a.w * sizeof(float));
  const size_t stage_bytes = tile_bytes_smem + kLabelBytes + ((zrow_bytes + 127u) & ~127u);
  auto stage_tile = [&](int s) { return reinterpret_cast<T*>(smem_raw + (size_t)s * stage_bytes); };
  auto stage_labels = [&](int s) {
    return reinterpret_cast<const int64_t*>(smem_raw + (size_t)s * stage_bytes + tile_bytes_smem);
  };
  auto stage_zrows = [&](int s) {
    return reinterpret_cast<float*>(smem_raw + (size_t)s * stage_bytes + tile_bytes_smem + kLabelBytes);
  };
  float2* strip = reinterpret_cast<float2*>(smem_raw + S * stage_bytes) + (size_t)wid * TH * kZCols;
  const int grid = (int)gridDim.x;
  const int my_tiles = (p.n_tiles - (int)blockIdx.x + grid - 1) / grid;
  const int tpi = p.tiles_per_image;

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&bar_full[s], 1);             // the loading lane's expect-tx arrival
      mbar_init(&bar_done[s], kFastThreads);  // every thread, after its gradient rows are written
    }
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();      // the seen logits, the labels and the logits come from the kernels before this one
  pdl_trigger();

  const int tiles_per_row = a.W / P;
  const bool tpr1 = tiles_per_row == 1;
  const int tpr_shift = (tiles_per_row & (tiles_per_row - 1)) == 0 ? __ffs(tiles_per_row) - 1 : -1;
  auto row_of_tile = [&](int t) { return tpr1 ? t : (tpr_shift >= 0 ? (t >> tpr_shift) : t / tiles_per_row); };
  // ---- TMA traffic.  Tile k of this CTA is OWNED by warp k % 8: its elected lane writes the gradient rows
  // back one iteration later (once every thread has arrived on bar_done) and, one iteration after that --
  // when its own store has drained the stage -- refills the stage with tile k + 4.  Every warp carries an
  // eighth of the issue work, none is a straggler, and a lane only ever waits on bulk groups it committed.
  auto tile_coords = [&](int k, int& b, int& t) {
    const int g = (int)blockIdx.x + k * grid;
    b = g / tpi;
    t = g - b * tpi;
  };
  auto slot_of = [](int k) { return k % S; };
  auto phase_of = [](int k) { return (uint32_t)((k / S) & 1); };
  const uint32_t tx_bytes = (uint32_t)K * (uint32_t)(P * sizeof(T)) + kLabelBytes + zrow_bytes;
  auto issue_load = [&](int k) {
    int b, t;
    tile_coords(k, b, t);
    const int s = slot_of(k);
    mbar_expect_tx(&bar_full[s], tx_bytes);
    T* dst = stage_tile(s);
    const Lerp ly = lerp_align_corners(row_of_tile(t), a.h, p.sy);
    tma_load_4d(stage_zrows(s), &p.tmap_z, 0, ly.i0, 0, b, &bar_full[s]);
    tma_load_3d(dst, &p.tmap_in, t * P, 0, b, &bar_full[s]);
    tma_load_3d(dst + (size_t)KREG * kBox, &p.tmap_in, t * P + kBox, 0, b, &bar_full[s]);
    bulk_g2s(const_cast<int64_t*>(stage_labels(s)), a.labels + (int64_t)b * HW + (int64_t)t * P, kLabelBytes,
             &bar_full[s]);
  };
  auto issue_store = [&](int k) {
    int b, t;
    tile_coords(k, b, t);
    const T* src = stage_tile(slot_of(k));
    tma_store_3d(&p.tmap_out, t * P, 0, b, src);
    tma_store_3d(&p.tmap_out, t * P + kBox, 0, b, src + (size_t)KREG * kBox);
    bulk_commit();
  };
  if (wid == 0 && elect_one()) {
    for (int k = 0; k < 2 && k < my_tiles; ++k) issue_load(k);
  }

  // tile geometry of the compute loop is advanced incrementally (no integer divisions)
  const int step_b = grid / tpi, step_t = grid - step_b * tpi;
  int tb = (int)blockIdx.x / tpi, tt = (int)blockIdx.x - tb * tpi;

  const int px0 = tid * 2;
  const int old_cl = min(max(a.old_cl, 1), K);
  const float u = (STD || a.ukd) ? 1.f : 0.f;
  const float gs_bacs = p.inv_n * a.grad_scale;
  const bool want_grad = a.dlogits != nullptr;
  const bool want_focal = a.gz != nullptr;
  float acc_loss = 0.f, acc_focal = 0.f;
  uint32_t cnt8 = 0;  // 8-bit fields: valid | invalid << 8 | bg << 16 | distill << 24
  uint32_t n_valid = 0, n_invalid = 0, n_bg = 0, n_dist = 0;
  auto flush_counts = [&]() {
    n_valid += cnt8 & 0xffu;
    n_invalid += (cnt8 >> 8) & 0xffu;
    n_bg += (cnt8 >> 16) & 0xffu;
    n_dist += cnt8 >> 24;
    cnt8 = 0;
  };

  // x geometry of this thread's two pixels; constant over the tiles when a tile is a whole image row
  int c_first = 0;       // first low-res column touched by the warp's 64 pixels
  int ci[2] = {0, 0};    // low-res column of each pixel relative to c_first (0..5)
  float wx1[2] = {0.f, 0.f};
  int gcol = 0;          // absolute low-res column of the first pixel of this lane's group of 8 lanes
  int gd[2] = {0, 0};    // column of each pixel relative to gcol (0 or 1)
  auto set_x = [&](int Xw) {
    c_first = lerp_align_corners(Xw, a.w, p.sx).i0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const Lerp lx = lerp_align_corners(Xw + 2 * lane + j, a.w, p.sx);
      ci[j] = lx.i0 - c_first;
      wx1[j] = lx.w1;
    }
    const int g0 = __shfl_sync(0xffffffffu, ci[0], lane & ~7);
    gcol = c_first + g0;
    gd[0] = ci[0] - g0;
    gd[1] = ci[1] - g0;
  };
  if (tpr1) set_x(wid * 64);

  for (int k = 0; k < my_tiles; ++k) {
    const int b = tb, t_in = tt;
    tb += step_b;
    tt += step_t;
    if (tt >= tpi) {
      tt -= tpi;
      ++tb;
    }
    const int s = slot_of(k);
    T* tile = stage_tile(s);
    const int Yrow = row_of_tile(t_in);
    const Lerp ly_row = lerp_align_corners(Yrow, a.h, p.sy);
    if (!tpr1) set_x((t_in - Yrow * tiles_per_row) * P + wid * 64);

    // ---- wait for the tile (logit rows + labels + seen-head rows) -------------------------------
    mbar_wait_sleepy(&bar_full[s], phase_of(k));
    const longlong2 lab = *reinterpret_cast<const longlong2*>(stage_labels(s) + px0);

    // ---- seen heads of this warp's 64 pixels: y-interpolated strip, stored per low-res column c as
    //      (z[c], z[c+1] - z[c]) so that the x-interpolation of a pixel is one LDS.64 + one FFMA ------
    {
      const float* zs = stage_zrows(s);
      const float wy1 = ly_row.w1, wy0 = 1.f - wy1;
      const int c = lane & (kZCols - 1);
      const int col = min(c_first + c, a.w - 1);
      const int r1 = (ly_row.i1 - ly_row.i0) * a.w;  // 0 on the last source row (the second TMA row is padding)
      __syncwarp();                                  // the previous tile's readers are done with the strip
      for (int t0 = 0; t0 < TH; t0 += 4) {           // uniform trip count: the shuffle needs the whole warp
        const int t = t0 + (lane >> 3);
        const float* zt = zs + (size_t)min(t, TH - 1) * 2 * a.w + col;
        const float v = __fadd_rn(__fmul_rn(wy0, zt[0]), __fmul_rn(wy1, zt[r1]));
        const float vn = __shfl_down_sync(0xffffffffu, v, 1);  // column c+1 (garbage for c == 7: never read)
        if (t < TH) strip[t * kZCols + c] = make_float2(v, vn - v);
      }
      __syncwarp();
    }

    // ---- labels -> class index (-1: ignore or invalid), counters ---------------------------------
    int y[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const long long l = j == 0 ? lab.x : lab.y;
      const bool ok = (unsigned long long)l < (unsigned long long)K;
      y[j] = ok ? (int)l : -1;
      cnt8 += ok ? (l == 0 ? 0x10001u : 1u) : (l != (long long)a.ignore_index ? 0x100u : 0u);
    }

    // ---- seen probability (max over heads of the up-sampled logits) and the focal head's logit ----
    float seen[2], zfoc[2] = {0.f, 0.f};
    {
      const float2* sp0 = strip + ci[0];
      const float2* sp1 = strip + ci[1];
      float zm0 = -INFINITY, zm1 = -INFINITY;
#pragma unroll
      for (int t = 0; t < 12; ++t) {
        if (t >= TH) break;
        const float2 v0 = sp0[t * kZCols], v1 = sp1[t * kZCols];
        zm0 = fmaxf(zm0, fmaf(wx1[0], v0.y, v0.x));
        zm1 = fmaxf(zm1, fmaf(wx1[1], v1.y, v1.x));
      }
      for (int t = 12; t < TH; ++t) {
        const float2 v0 = sp0[t * kZCols], v1 = sp1[t * kZCols];
        zm0 = fmaxf(zm0, fmaf(wx1[0], v0.y, v0.x));
        zm1 = fmaxf(zm1, fmaf(wx1[1], v1.y, v1.x));
      }
      seen[0] = rcp_fast(1.f + ex2_fast(-kLog2e * zm0));
      seen[1] = rcp_fast(1.f + ex2_fast(-kLog2e * zm1));
      if (want_focal) {
        const float2 v0 = sp0[a.focal_head * kZCols], v1 = sp1[a.focal_head * kZCols];
        zfoc[0] = fmaf(wx1[0], v0.y, v0.x);
        zfoc[1] = fmaf(wx1[1], v1.y, v1.x);
      }
    }

    // ---- registers <- shared memory; max / arg-max on the packed pair ------------------------------
    // pixel pair 2*tid lives in box tid/128 at column (2*tid) % 256; channel rows are kBox apart
    T* col = tile + (size_t)(tid >> 7) * KREG * kBox + ((2 * tid) & (kBox - 1));
    float xy[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) xy[j] = (y[j] >= old_cl) ? DT<T>::to_f(col[(size_t)y[j] * kBox + j]) : 0.f;
    typename Raw<T>::reg_t raw[KREG];
#pragma unroll
    for (int c = 0; c < KREG; ++c) {
      if (c < KMIN || c < K) raw[c] = Raw<T>::ld(col + (size_t)c * kBox);
      else raw[c] = NegInf<T>::pair();
    }
    typename Raw<T>::Max mt = Raw<T>::init(raw[0]);
#pragma unroll
    for (int c = 1; c < KREG; ++c) Raw<T>::update(mt, raw[c], c);
    float mx0, mx1;
    int am0, am1;
    Raw<T>::finish(mt, mx0, mx1, am0, am1);

    // ---- one exp per logit; sums in groups of four so that S_old costs one add per full group.  The two pixels
    //      of a thread travel as one packed fp32 pair (FFMA2 / FADD2): half the issue slots of the scalar form ------
    const float nm0 = -mx0 * kLog2e, nm1 = -mx1 * kLog2e;
    const F2 nm2 = f2(nm0, nm1), l2e2 = f2b(kLog2e);
    F2 e2[KREG];
    F2 sa2 = f2b(0.f), so2 = f2b(0.f);
    float x00, x01;
    Raw<T>::unpack(raw[0], x00, x01);
#pragma unroll
    for (int g = 0; g < (KREG + 3) / 4; ++g) {
      F2 g2 = f2b(0.f);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = 4 * g + i;
        if (c < KREG) {
          float v0, v1;
          Raw<T>::unpack(raw[c], v0, v1);
          const F2 arg = fma2(f2(v0, v1), l2e2, nm2);
          e2[c] = f2(ex2_fast(f2lo(arg)), ex2_fast(f2hi(arg)));
          if (c >= 1) g2 = (i == 0 || c == 1) ? e2[c] : add2(g2, e2[c]);  // channel 0 is kept out of the sums
        }
      }
      sa2 = add2(sa2, g2);
      if (4 * g + 4 <= old_cl) {  // uniform: the whole group is old
        so2 = add2(so2, g2);
      } else if (4 * g < old_cl) {  // uniform: the boundary group
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int c = 4 * g + i;
          if (c >= 1 && c < KREG && c < old_cl) so2 = add2(so2, e2[c]);
        }
      }
    }
    // S_fg = sum_{c>=1} is accumulated directly (S - e_0 would cancel when the background logit dominates);
    // S = S_fg + e_0, S_old = e_0 + sum_{1<=c<old_cl}
    const float sf0 = f2lo(sa2), sf1 = f2hi(sa2);
    sa2 = add2(sa2, e2[0]);
    so2 = add2(so2, e2[0]);
    const float sa0 = f2lo(sa2), sa1 = f2hi(sa2), so0 = f2lo(so2), so1 = f2hi(so2);

    // ---- per-pixel terms: loss, gradient coefficients, distill mask, focal term (select-only) ------
    //   gradient of pixel = e_c * cg[group(c)] - [c==0] d0 - [c==y] dy,  groups: c == 0 | 1 <= c < old_cl | c >= old_cl
    float cg0[2], cg1[2], cg2[2], d0[2], dy[2], gfoc[2];
    uint32_t dmask2 = 0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float mx = j == 0 ? mx0 : mx1, Sa = j == 0 ? sa0 : sa1, So = fmaxf(j == 0 ? so0 : so1, 1e-37f);
      const float ec0 = j == 0 ? f2lo(e2[0]) : f2hi(e2[0]), x0 = j == 0 ? x00 : x01;
      const bool valid = y[j] >= 0, isbg = y[j] == 0, isnew = y[j] >= old_cl;
      const float Sfg = fmaxf(j == 0 ? sf0 : sf1, 1e-37f);
      const float lS = lg2_fast(Sa), iS = rcp_fast(Sa);
      const float lF = lg2_fast(Sfg), iF = rcp_fast(Sfg);
      float lO = 0.f, iO = 0.f;
      if (STD || a.ukd) {  // uniform
        lO = lg2_fast(So);
        iO = rcp_fast(So);
      }
      const float sm = seen[j] > a.threshold ? 1.f : seen[j];
      const float mod = STD ? (1.f - sm) * (1.f - sm) : pow_gamma(1.f - sm, a.gamma);
      const float m = isbg ? mod : 1.f;
      const float uo = isnew ? 0.f : u;
      const float a1 = m + (isnew ? 1.f : uo);
      const float f = isbg ? 0.f : iF;
      const float gsv = valid ? gs_bacs : 0.f;
      const float c0 = fmaf(a1, iS, -uo * iO);
      cg0[j] = c0 * gsv;
      cg1[j] = (c0 - f) * gsv;
      cg2[j] = fmaf(a1, iS, -f) * gsv;
      d0[j] = isbg ? mod * gsv : 0.f;
      dy[j] = isnew ? gsv : 0.f;
      const float lseS = kLn2 * lS;
      const float t1 = isbg ? mod * (mx - x0 + lseS) : kLn2 * (lS - lF);
      const float t2 = isnew ? (mx - xy[j] + lseS) : u * kLn2 * (lS - lO);
      acc_loss += valid ? t1 + t2 : 0.f;
      const bool dm = isbg && seen[j] > a.lkd_threshold;
      dmask2 |= dm ? (1u << (8 * j)) : 0u;
      cnt8 += dm ? 0x1000000u : 0u;
      gfoc[j] = 0.f;
      if (want_focal) {  // uniform
        float term, dterm;
        if (STD) {
          // binary focal loss, gamma = 2, target t = foreground: bce = softplus(Z) - t Z, pt = exp(-bce)
          const float Z = zfoc[j];
          const float e = ex2_fast(-kLog2e * fabsf(Z));
          const float d = 1.f + e;
          const float hi = rcp_fast(d), lo = e * hi;      // sigmoid(|Z|), sigmoid(-|Z|)
          const float l1p = kLn2 * lg2_fast(d);
          const bool pos = Z >= 0.f;
          const float sig = pos ? hi : lo, nsig = pos ? lo : hi;
          const float pt = isbg ? nsig : sig, om = isbg ? sig : nsig;
          const float bce = fmaxf(Z, 0.f) - (isbg ? 0.f : Z) + l1p;
          const float om2 = om * om;
          term = om2 * bce;
          dterm = (isbg ? sig : -nsig) * fmaf(2.f * om * pt, bce, om2);
        } else {
          focal_term(a, zfoc[j], isbg ? 0.f : 1.f, term, dterm);
        }
        acc_focal += valid ? term : 0.f;
        gfoc[j] = valid ? dterm : 0.f;
      }
    }

    // ---- gradient rows, in place ----------------------------------------------------------------------------
    if (want_grad) {
      const F2 cgo = f2(cg1[0], cg1[1]), cgn = f2(cg2[0], cg2[1]);  // old / new class coefficient of both pixels
      {
        const F2 g0 = fma2(e2[0], f2(cg0[0], cg0[1]), f2(-d0[0], -d0[1]));
        Raw<T>::st(col, f2lo(g0), f2hi(g0));
      }
#pragma unroll
      for (int g = 0; g < (KREG + 3) / 4; ++g) {
        if (4 * g + 4 <= old_cl) {  // uniform: old classes only
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int c = 4 * g + i;
            if (c >= 1 && c < KREG) {
              const F2 gg = mul2(e2[c], cgo);
              Raw<T>::st(col + (size_t)c * kBox, f2lo(gg), f2hi(gg));
            }
          }
        } else if (4 * g >= old_cl) {  // uniform: new classes only
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int c = 4 * g + i;
            if (c >= 1 && c < KREG) {
              const F2 gg = mul2(e2[c], cgn);
              Raw<T>::st(col + (size_t)c * kBox, f2lo(gg), f2hi(gg));
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int c = 4 * g + i;
            if (c >= 1 && c < KREG) {
              const F2 gg = mul2(e2[c], c < old_cl ? cgo : cgn);
              Raw<T>::st(col + (size_t)c * kBox, f2lo(gg), f2hi(gg));
            }
          }
        }
      }
      // a new-class label's own channel: recomputed in fp32 so that -dy is applied before rounding
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (y[j] >= old_cl) {
          const float ey = ex2_fast(fmaf(xy[j], kLog2e, j == 0 ? nm0 : nm1));
          col[(size_t)y[j] * kBox + j] = DT<T>::from_f(fmaf(ey, cg2[j], -dy[j]));
        }
      }
      fence_proxy_async();
    }
    mbar_arrive(&bar_done[s]);

    // ---- tile owners: write tile k-1 back; refill a drained stage with tile k+2 ---------------------------
    // 4 stages: tile k+2 goes into the stage of tile k-2, whose owner stored it one iteration ago.
    // 3 stages (when two CTAs per SM only fit that way): tile k+2 goes into the stage of tile k-1, so its owner
    // stores, waits for the store to have read the stage, and reloads in the same visit.
    if (k >= 1 && wid == ((k - 1) & 7)) {
      if (elect_one()) {
        mbar_wait(&bar_done[slot_of(k - 1)], phase_of(k - 1));  // gradients of tile k-1 written
        if (want_grad) issue_store(k - 1);
        if (S == 3) {
          if (want_grad) bulk_wait_read0();
          if (k + 2 < my_tiles) issue_load(k + 2);
        }
      }
      __syncwarp();
    }
    if (S == 4 && wid == ((k + 6) & 7)) {
      if (elect_one()) {
        // this lane waited for bar_done of tile k-2 one iteration ago; its store has had a tile to drain
        if (want_grad) bulk_wait_read0();
        if (k + 2 < my_tiles) issue_load(k + 2);
      }
      __syncwarp();
    }
    if (S == 3 && k == 0 && wid == 7) {  // the third stage is still fresh: nothing to drain
      if (elect_one() && 2 < my_tiles) issue_load(2);
      __syncwarp();
    }

    // ---- arg-max / mask stores -------------------------------------------------------------------------
    const int64_t pix = (int64_t)b * HW + (int64_t)t_in * P + px0;
    if (a.preds) *reinterpret_cast<longlong2*>(a.preds + pix) = make_longlong2((long long)am0, (long long)am1);
    if (a.distill_mask) *reinterpret_cast<uint16_t*>(a.distill_mask + pix) = (uint16_t)dmask2;

    // ---- focal gradient: adjoint of the bilinear up-sample ---------------------------------------------
    // The 16 pixels of a group of 8 lanes touch the low-res columns gcol, gcol+1, gcol+2 only.
    if (want_focal) {
      const unsigned full = 0xffffffffu;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float hi = gfoc[j] * wx1[j], lo = gfoc[j] - hi;  // weights wx1 and 1 - wx1
        if (gd[j] == 0) {
          s0 += lo;
          s1 += hi;
        } else {
          s1 += lo;
          s2 += hi;
        }
      }
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        s0 += __shfl_xor_sync(full, s0, o);
        s1 += __shfl_xor_sync(full, s1, o);
        s2 += __shfl_xor_sync(full, s2, o);
      }
      const int r = lane & 7;  // lanes 0..2: upper source row, 3..5: lower source row
      if (r < 6) {
        const int cc = r >= 3 ? r - 3 : r;
        const float sv = cc == 0 ? s0 : (cc == 1 ? s1 : s2);
        const float wy = r >= 3 ? ly_row.w1 : 1.f - ly_row.w1;
        const float val = sv * wy;
        const int row = r >= 3 ? ly_row.i1 : ly_row.i0;
        if (val != 0.f) atomicAdd(a.gz + ((int64_t)b * a.h + row) * a.w + min(gcol + cc, a.w - 1), val);
      }
    }
    if ((k & 63) == 63) flush_counts();
  }
  if (my_tiles > 0) {  // the last tile's gradient rows; every lane that committed bulk stores drains them
    const int kl = my_tiles - 1;
    if (elect_one()) {
      if (wid == (kl & 7)) {
        mbar_wait(&bar_done[slot_of(kl)], phase_of(kl));
        if (want_grad) issue_store(kl);
      }
      bulk_wait_all();
    }
    __syncwarp();
  }

  flush_counts();
  float acc[BACS_NACC];
  acc[BACS_ACC_LOSS] = acc_loss;
  acc[BACS_ACC_WSUM] = 0.f;
  acc[BACS_ACC_FOCAL] = acc_focal;
  acc[BACS_ACC_KEPT] = (float)n_valid;
  acc[BACS_ACC_BG] = (float)n_bg;
  acc[BACS_ACC_INVALID] = (float)n_invalid;
  acc[BACS_ACC_DISTILL_PIX] = (float)n_dist;
  acc[BACS_ACC_VALID] = (float)n_valid;
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) {
    const float r = warp_sum(acc[i]);
    if (lane == 0) red_scratch[wid][i] = r;
  }
  __syncthreads();
  if (tid < BACS_NACC) {
    double r = 0.0;
    for (int wv = 0; wv < 8; ++wv) r += (double)red_scratch[wv][tid];
    p.partials[(int64_t)blockIdx.x * BACS_NACC + tid] = r;
  }
}

template <typename T, int KREG>
static int launch_wce_one(const PixelParams& p, const PixelPlan& plan, cudaStream_t s) {
  const bacs_pixel_args& a = p.a;
  const bool std_hp = a.gamma == 2.f && a.ukd && (!a.gz || (a.focal_gamma == 2.f && a.focal_alpha < 0.f));
  auto kern = plan.stages == 3 ? (std_hp ? pixel_wce_kernel<T, KREG, true, 3> : pixel_wce_kernel<T, KREG, false, 3>)
                               : (std_hp ? pixel_wce_kernel<T, KREG, true, 4> : pixel_wce_kernel<T, KREG, false, 4>);
  return launch_pixel_kernel("bacs_pixel_loss", true, kern, dim3(plan.grid), dim3(kFastThreads), plan.smem, s, p);
}

template <typename T>
static int launch_wce_dtype(const PixelParams& p, const PixelPlan& plan, cudaStream_t s) {
  switch (plan.kreg) {
    case 4: return launch_wce_one<T, 4>(p, plan, s);
    case 8: return launch_wce_one<T, 8>(p, plan, s);
    case 12: return launch_wce_one<T, 12>(p, plan, s);
    case 16: return launch_wce_one<T, 16>(p, plan, s);
    case 20: return launch_wce_one<T, 20>(p, plan, s);
    case 21: return launch_wce_one<T, 21>(p, plan, s);
    case 24: return launch_wce_one<T, 24>(p, plan, s);
    default:
      set_error("bacs_pixel_loss: no training-step kernel for KREG=%d", plan.kreg);
      return BACS_ERR_UNSUPPORTED;
  }
}

}  // namespace bacs
