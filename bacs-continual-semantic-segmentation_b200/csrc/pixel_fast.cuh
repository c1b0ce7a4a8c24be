// Register-resident fast path of the fused per-pixel kernel (K <= 24, even image sizes,
// 16-byte aligned rows).  Included by one translation unit per storage type.
//
// Persistent CTAs of 8 warps; every thread owns 2 adjacent pixels of a 512-pixel tile.
// A 4-stage TMA ring moves the tiles: one elected lane issues, per tile, two 3-D tiled TMA
// loads (tensor map (H*W, K, B), box 256 x K x 1: all K logit rows of 256 pixels in ONE
// instruction), one bulk copy of the tile's 4 KB label strip, and two tiled TMA stores of the
// gradient.  While tile k is computed, tile k+1 has landed, tile k+2 is landing into the
// stage of tile k-2 and tile k-1 is being written back, so the issuing lane never blocks and
// there is no CTA-wide barrier in the tile loop.  The K logits of both pixels live in
// registers from the single shared-memory read to the gradient write (one exp per logit).
#pragma once
#include "pixel_common.cuh"

namespace bacs {

constexpr int kFastThreads = 256;
constexpr int kFastP = 512;

// Two adjacent pixels of one channel row, as they sit in shared memory, plus the running
// (max, arg-max) of both pixels.  For the 16-bit types the maximum and the arg-max are
// tracked on the PACKED pair (HMNMX2 + HSET2 mask + LOP3): 3 instructions per channel
// for both pixels; ties keep the lowest channel (strict >), as torch.argmax does.
template <typename T> struct Raw;
template <> struct Raw<float> {
  using reg_t = float2;
  struct Max {
    float m0, m1;
    int a0, a1;
  };
  __device__ static __forceinline__ reg_t ld(const float* p) { return *reinterpret_cast<const float2*>(p); }
  __device__ static __forceinline__ void st(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
  __device__ static __forceinline__ void fill(float* p, float v) { *p = v; }
  __device__ static __forceinline__ void unpack(reg_t r, float& a, float& b) { a = r.x; b = r.y; }
  __device__ static __forceinline__ Max init(reg_t r) { return Max{r.x, r.y, 0, 0}; }
  __device__ static __forceinline__ void set_first(Max& m, int c) { m.a0 = m.a1 = c; }
  __device__ static __forceinline__ void update(Max& m, reg_t r, int c) {
    if (r.x > m.m0) { m.m0 = r.x; m.a0 = c; }
    if (r.y > m.m1) { m.m1 = r.y; m.a1 = c; }
  }
  __device__ static __forceinline__ void finish(const Max& m, float& m0, float& m1, int& a0, int& a1) {
    m0 = m.m0; m1 = m.m1; a0 = m.a0; a1 = m.a1;
  }
};
template <> struct Raw<__nv_bfloat16> {
  using reg_t = uint32_t;
  struct Max {
    __nv_bfloat162 m;
    uint32_t a;
  };
  __device__ static __forceinline__ reg_t ld(const __nv_bfloat16* p) { return *reinterpret_cast<const uint32_t*>(p); }
  __device__ static __forceinline__ void st(__nv_bfloat16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
  }
  __device__ static __forceinline__ void fill(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  __device__ static __forceinline__ void unpack(reg_t u, float& a, float& b) {
    a = __uint_as_float(u << 16);
    b = __uint_as_float(u & 0xffff0000u);
  }
  __device__ static __forceinline__ Max init(reg_t r) { return Max{*reinterpret_cast<__nv_bfloat162*>(&r), 0u}; }
  __device__ static __forceinline__ void set_first(Max& m, int c) { m.a = (uint32_t)c | ((uint32_t)c << 16); }
  __device__ static __forceinline__ void update(Max& m, reg_t r, int c) {
    const __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&r);
    const uint32_t mask = __hgt2_mask(v, m.m);
    m.m = __hmax2(v, m.m);
    const uint32_t cc = (uint32_t)c | ((uint32_t)c << 16);
    m.a = (m.a & ~mask) | (cc & mask);
  }
  __device__ static __forceinline__ void finish(const Max& m, float& m0, float& m1, int& a0, int& a1) {
    const float2 f = __bfloat1622float2(m.m);
    m0 = f.x; m1 = f.y;
    a0 = (int)(m.a & 0xffffu); a1 = (int)(m.a >> 16);
  }
};
template <> struct Raw<__half> {
  using reg_t = uint32_t;
  struct Max {
    __half2 m;
    uint32_t a;
  };
  __device__ static __forceinline__ reg_t ld(const __half* p) { return *reinterpret_cast<const uint32_t*>(p); }
  __device__ static __forceinline__ void st(__half* p, float a, float b) {
    *reinterpret_cast<__half2*>(p) = __floats2half2_rn(a, b);
  }
  __device__ static __forceinline__ void fill(__half* p, float v) { *p = __float2half_rn(v); }
  __device__ static __forceinline__ void unpack(reg_t u, float& a, float& b) {
    const float2 f = __half22float2(*reinterpret_cast<__half2*>(&u));
    a = f.x; b = f.y;
  }
  __device__ static __forceinline__ Max init(reg_t r) { return Max{*reinterpret_cast<__half2*>(&r), 0u}; }
  __device__ static __forceinline__ void set_first(Max& m, int c) { m.a = (uint32_t)c | ((uint32_t)c << 16); }
  __device__ static __forceinline__ void update(Max& m, reg_t r, int c) {
    const __half2 v = *reinterpret_cast<__half2*>(&r);
    const uint32_t mask = __hgt2_mask(v, m.m);
    m.m = __hmax2(v, m.m);
    const uint32_t cc = (uint32_t)c | ((uint32_t)c << 16);
    m.a = (m.a & ~mask) | (cc & mask);
  }
  __device__ static __forceinline__ void finish(const Max& m, float& m0, float& m1, int& a0, int& a1) {
    const float2 f = __half22float2(m.m);
    m0 = f.x; m1 = f.y;
    a0 = (int)(m.a & 0xffffu); a1 = (int)(m.a >> 16);
  }
};

__device__ __forceinline__ void fast_sync() { __syncthreads(); }

constexpr int kZCols = 8;          // low-res columns a warp's 64 pixels can touch (x16 up-sampling: <= 6)
constexpr int kLabelBytes = kFastP * 8;

// Shared memory (dynamic): 4 stages of { [2][KREG][256] logits -- two TMA boxes of 256 pixels; rows
// K..KREG-1 of each box hold -inf forever --, 512 int64 labels } followed by one warp-private
// [T][kZCols] seen-logit strip per warp.
constexpr int kBox = 256;
template <typename T, int KREG, bool ROWTILE>
__global__ void __launch_bounds__(kFastThreads, 2) pixel_fast_kernel(const __grid_constant__ PixelParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t bar_full[4];
  __shared__ uint64_t bar_done[4];
  __shared__ float red_scratch[8][BACS_NACC];
  __shared__ float s_norm_sh;

  constexpr int P = kFastP, S = 4;
  constexpr size_t tile_elems = (size_t)KREG * P;
  const bacs_pixel_args& a = p.a;
  // per stage: logits | labels | (row tiles) the two source rows of every seen head, [T][2][w] fp32
  const uint32_t zrow_bytes = (ROWTILE && a.z) ? (uint32_t)(a.T * 2 * a.w * sizeof(float)) : 0u;
  const size_t stage_bytes = tile_elems * sizeof(T) + kLabelBytes + ((zrow_bytes + 127u) & ~127u);
  const int K = a.K;
  const int tid = threadIdx.x;
  const int lane = tid & 31, wid = tid >> 5;
  const int64_t HW = (int64_t)a.H * a.W;
  auto stage_tile = [&](int s) { return reinterpret_cast<T*>(smem_raw + (size_t)s * stage_bytes); };
  auto stage_labels = [&](int s) {
    return reinterpret_cast<const int64_t*>(smem_raw + (size_t)s * stage_bytes + tile_elems * sizeof(T));
  };
  auto stage_zrows = [&](int s) {
    return reinterpret_cast<float*>(smem_raw + (size_t)s * stage_bytes + tile_elems * sizeof(T) + kLabelBytes);
  };
  float* zrw = reinterpret_cast<float*>(smem_raw + S * stage_bytes) + (size_t)wid * a.T * kZCols;
  const int grid = (int)gridDim.x;
  const int my_tiles = (p.n_tiles - (int)blockIdx.x + grid - 1) / grid;
  const int tpi = p.tiles_per_image;
  const uint32_t row_bytes = (uint32_t)(P * sizeof(T));

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&bar_full[s], 1);             // the issuing lane's expect-tx arrival
      mbar_init(&bar_done[s], kFastThreads);  // every thread, after its gradient rows are written
    }
    fence_mbar_init();
    s_norm_sh = 0.f;
  }
  // padding rows stay -inf: exp -> 0, never the arg-max, never stored
  for (int i = tid; i < S * 2 * (KREG - K) * kBox; i += kFastThreads) {
    const int sb2 = i / ((KREG - K) * kBox), r = i - sb2 * (KREG - K) * kBox;  // sb2 = stage*2 + box
    Raw<T>::fill(stage_tile(sb2 >> 1) + (size_t)(sb2 & 1) * KREG * kBox + (size_t)K * kBox + r, -INFINITY);
  }
  __syncthreads();
  if (tid < 32 && a.mode != BACS_PIX_WEIGHTED_CE && a.dlogits != nullptr) {
    double s = 0.0;
    for (int c = tid; c < K && c < 256; c += 32)
      if (c != a.ignore_index)
        s += (double)a.hist[c] * ((a.mode == BACS_PIX_CE && a.class_w) ? (double)a.class_w[c] : 1.0);
    s = warp_sum(s);
    if (tid == 0) s_norm_sh = s > 0.0 ? (float)(1.0 / s) : 0.f;
  }
  __syncthreads();

  // tile geometry is advanced incrementally (no integer divisions in the loop)
  const int step_b = grid / tpi, step_t = grid - step_b * tpi;
  int tb = (int)blockIdx.x / tpi, tt = (int)blockIdx.x - tb * tpi;  // tile k of this CTA: image tb, tile tt
  auto advance = [&](int& b, int& t) {
    b += step_b;
    t += step_t;
    if (t >= tpi) {
      t -= tpi;
      ++b;
    }
  };
  // one elected lane of warp 0 issues all TMA traffic of the CTA (5 instructions per tile)
  const uint32_t tile_bytes = (uint32_t)K * row_bytes + kLabelBytes + zrow_bytes;
  const int tiles_per_row = ROWTILE ? a.W / P : 1;
  const int tpr_shift = (tiles_per_row & (tiles_per_row - 1)) == 0 ? __ffs(tiles_per_row) - 1 : -1;
  auto row_of_tile = [&](int t) { return tpr_shift >= 0 ? (t >> tpr_shift) : t / tiles_per_row; };
  auto issue_load = [&](int b, int t, int s) {
    mbar_expect_tx(&bar_full[s], tile_bytes);
    T* dst = stage_tile(s);
    if (ROWTILE && a.z) {  // rows i0, i0+1 of all T heads for the image row this tile lies in
      const Lerp ly = lerp_align_corners(row_of_tile(t), a.h, p.sy);
      if (p.use_tmap) {
        tma_load_4d(stage_zrows(s), &p.tmap_z, 0, ly.i0, 0, b, &bar_full[s]);
      } else {
        const float* zb = a.z + (int64_t)b * a.T * a.h * a.w;
        for (int h2 = 0; h2 < a.T; ++h2) {
          bulk_g2s(stage_zrows(s) + (size_t)(2 * h2) * a.w, zb + ((int64_t)h2 * a.h + ly.i0) * a.w,
                   (uint32_t)(a.w * sizeof(float)), &bar_full[s]);
          bulk_g2s(stage_zrows(s) + (size_t)(2 * h2 + 1) * a.w, zb + ((int64_t)h2 * a.h + ly.i1) * a.w,
                   (uint32_t)(a.w * sizeof(float)), &bar_full[s]);
        }
      }
    }
    if (p.use_tmap) {
      tma_load_3d(dst, &p.tmap_in, t * P, 0, b, &bar_full[s]);
      tma_load_3d(dst + (size_t)KREG * kBox, &p.tmap_in, t * P + kBox, 0, b, &bar_full[s]);
    } else {  // driver without tensor-map support: 2K one-dimensional bulk copies
      const T* src = reinterpret_cast<const T*>(a.logits) + (int64_t)b * K * HW + (int64_t)t * P;
      for (int c = 0; c < K; ++c) {
        bulk_g2s(dst + (size_t)c * kBox, src + (int64_t)c * HW, row_bytes / 2, &bar_full[s]);
        bulk_g2s(dst + (size_t)(KREG + c) * kBox, src + (int64_t)c * HW + kBox, row_bytes / 2, &bar_full[s]);
      }
    }
    bulk_g2s(const_cast<int64_t*>(stage_labels(s)), a.labels + (int64_t)b * HW + (int64_t)t * P, kLabelBytes,
             &bar_full[s]);
  };
  auto issue_store = [&](int b, int t, int s) {
    const T* src = stage_tile(s);
    if (p.use_tmap) {
      tma_store_3d(&p.tmap_out, t * P, 0, b, src);
      tma_store_3d(&p.tmap_out, t * P + kBox, 0, b, src + (size_t)KREG * kBox);
    } else {
      T* dst = reinterpret_cast<T*>(a.dlogits) + (int64_t)b * K * HW + (int64_t)t * P;
      for (int c = 0; c < K; ++c) {
        bulk_s2g(dst + (int64_t)c * HW, src + (size_t)c * kBox, row_bytes / 2);
        bulk_s2g(dst + (int64_t)c * HW + kBox, src + (size_t)(KREG + c) * kBox, row_bytes / 2);
      }
    }
    bulk_commit();
  };
  int pb = tb, pt = tt;  // load cursor (tile k + 2)
  int sb = tb, st = tt;  // store cursor (tile k - 1)
  bool issuer = false;   // the elected lane of warp 0 (the same lane every time: bulk groups are per thread)
  if (wid == 0) issuer = elect_one();
  if (issuer) {
    for (int k = 0; k < 2 && k < my_tiles; ++k) {
      issue_load(pb, pt, k);
      advance(pb, pt);
    }
  }

  const int px0 = tid * 2;
  const int old_cl = min(max(a.old_cl, 0), K);
  const bool have_seen = (a.z != nullptr) || (a.seen_max != nullptr);
  const float s_norm = s_norm_sh;
  float acc[BACS_NACC];
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) acc[i] = 0.f;
  // x-interpolation of this thread's two pixels; constant over tiles when a tile is a whole row
  Lerp lxj[2] = {{0, 0, 0.f}, {0, 0, 0.f}};
  int c_first = 0;

  for (int k = 0; k < my_tiles; ++k) {
    const int b = tb, t_in = tt;
    advance(tb, tt);
    const int s = k % S;
    const uint32_t parity = (uint32_t)((k / S) & 1);
    T* tile = stage_tile(s);
    const int64_t p0 = (int64_t)t_in * P;

    // ---- wait for the tile (logit rows + labels + seen-head rows) -------------------------------
    mbar_wait(&bar_full[s], parity);
    const longlong2 lab = *reinterpret_cast<const longlong2*>(stage_labels(s) + px0);

    // ---- seen logits of this warp's 64 pixels: y-interpolated strip in warp-private smem ------
    Lerp ly_row = {0, 0, 0.f};
    if (ROWTILE && a.z) {
      const int Yrow = row_of_tile(t_in);
      ly_row = lerp_align_corners(Yrow, a.h, p.sy);
      if (k == 0 || tiles_per_row != 1) {
        const int Xw = (t_in - Yrow * tiles_per_row) * P + wid * 64;
        c_first = lerp_align_corners(Xw, a.w, p.sx).i0;
        lxj[0] = lerp_align_corners(Xw + 2 * lane, a.w, p.sx);
        lxj[1] = lerp_align_corners(Xw + 2 * lane + 1, a.w, p.sx);
      }
      const float* zs = stage_zrows(s);
      const float wy0 = 1.f - ly_row.w1;
      const int col = min(c_first + (lane & (kZCols - 1)), a.w - 1);
      const int r1 = (ly_row.i1 - ly_row.i0) * a.w;  // 0 on the last source row (the second TMA row is padding)
      __syncwarp();
      for (int t = lane / kZCols; t < a.T; t += 32 / kZCols) {
        const float* zt = zs + (size_t)t * 2 * a.w + col;
        zrw[t * kZCols + (lane & (kZCols - 1))] = __fadd_rn(__fmul_rn(wy0, zt[0]), __fmul_rn(ly_row.w1, zt[r1]));
      }
      __syncwarp();
    }

    int y[2];
    bool is_ign[2];
    float seen[2], zfoc[2], wx1[2];
    int cx0[2], cdx[2];
    int cell[2], cell_dy[2];
    float wy1g[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int64_t l = j == 0 ? lab.x : lab.y;
      y[j] = -1;
      is_ign[j] = true;
      seen[j] = zfoc[j] = wx1[j] = wy1g[j] = 0.f;
      cx0[j] = cell[j] = -1;
      cdx[j] = cell_dy[j] = 0;
      if (l == a.ignore_index) {
      } else if (l >= 0 && l < K) {
        y[j] = (int)l;
        is_ign[j] = false;
      } else {
        acc[BACS_ACC_INVALID] += 1.f;
      }
      if (a.seen_max) seen[j] = __ldg(a.seen_max + (int64_t)b * HW + p0 + px0 + j);
      if (a.z) {
        float zmax = -INFINITY;
        if (ROWTILE) {
          const Lerp lx = lxj[j];
          const float wx0 = 1.f - lx.w1;
          const float* z0 = zrw + (lx.i0 - c_first);
          const int dx = lx.i1 - lx.i0;
          for (int t = 0; t < a.T; ++t) {
            const float v = __fadd_rn(__fmul_rn(wx0, z0[t * kZCols]), __fmul_rn(lx.w1, z0[t * kZCols + dx]));
            zmax = fmaxf(zmax, v);
            if (t == a.focal_head) zfoc[j] = v;
          }
          cx0[j] = lx.i0;
          cdx[j] = dx;
          wx1[j] = lx.w1;
        } else {
          const int64_t pix = p0 + px0 + j;
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

    // ---- registers <- shared memory; max / arg-max on the packed pair ------------------------------
    // pixel pair 2*tid lives in box tid/128 at column (2*tid) % 256; channel rows are kBox apart
    T* col = tile + (size_t)(tid >> 7) * KREG * kBox + ((2 * tid) & (kBox - 1));
    float xy[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) xy[j] = (y[j] >= 0) ? DT<T>::to_f(col[(size_t)y[j] * kBox + j]) : 0.f;
    typename Raw<T>::reg_t raw[KREG];
#pragma unroll
    for (int c = 0; c < KREG; ++c) raw[c] = Raw<T>::ld(col + (size_t)c * kBox);
    typename Raw<T>::Max mt = Raw<T>::init(raw[0]);
#pragma unroll
    for (int c = 1; c < KREG; ++c) Raw<T>::update(mt, raw[c], c);
    float mx0, mx1;
    int am0, am1;
    Raw<T>::finish(mt, mx0, mx1, am0, am1);

    // ---- one exp per logit; sums in groups of four so that S_old costs one add per full group ------
    const float nm0 = -mx0 * kLog2e, nm1 = -mx1 * kLog2e;
    float e0[KREG], e1[KREG];
    float sa0 = 0.f, sa1 = 0.f, so0 = 0.f, so1 = 0.f;
    float x00, x01;
    Raw<T>::unpack(raw[0], x00, x01);
#pragma unroll
    for (int g = 0; g < (KREG + 3) / 4; ++g) {
      float g0 = 0.f, g1 = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = 4 * g + i;
        if (c < KREG) {
          float v0, v1;
          Raw<T>::unpack(raw[c], v0, v1);
          e0[c] = ex2_fast(fmaf(v0, kLog2e, nm0));
          e1[c] = ex2_fast(fmaf(v1, kLog2e, nm1));
          if (c >= 1) {  // channel 0 is kept out of the sums: S_fg is accumulated directly
            g0 = (i == 0 || c == 1) ? e0[c] : g0 + e0[c];
            g1 = (i == 0 || c == 1) ? e1[c] : g1 + e1[c];
          }
        }
      }
      sa0 += g0;
      sa1 += g1;
      if (4 * g + 4 <= old_cl) {  // uniform: the whole group is old
        so0 += g0;
        so1 += g1;
      } else if (4 * g < old_cl) {  // uniform: the boundary group
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int c = 4 * g + i;
          if (c >= 1 && c < KREG && c < old_cl) {
            so0 += e0[c];
            so1 += e1[c];
          }
        }
      }
    }

    // S_fg = sum_{c>=1} (accumulated above), S = S_fg + e_0, S_old = [old_cl >= 1] e_0 + sum_{1<=c<old_cl}
    const float sf0 = sa0, sf1 = sa1;
    sa0 += e0[0];
    sa1 += e1[0];
    if (old_cl >= 1) {
      so0 += e0[0];
      so1 += e1[0];
    }
    PixCoef pc[2];
    float gfoc[2];
    uint8_t dmask[2];
    pixel_terms(a, p.inv_n, s_norm, old_cl, y[0], is_ign[0], mx0, sa0, so0, sf0, e0[0], x00, xy[0], seen[0], have_seen,
                zfoc[0], acc, pc[0], gfoc[0], dmask[0]);
    pixel_terms(a, p.inv_n, s_norm, old_cl, y[1], is_ign[1], mx1, sa1, so1, sf1, e1[0], x01, xy[1], seen[1], have_seen,
                zfoc[1], acc, pc[1], gfoc[1], dmask[1]);
    if (a.dlogits) {
      Raw<T>::st(col, e0[0] * pc[0].cg0 - pc[0].d0, e1[0] * pc[1].cg0 - pc[1].d0);
#pragma unroll
      for (int c = 1; c < KREG; ++c) {
        const bool oldc = c < old_cl;
        const float g0 = e0[c] * (oldc ? pc[0].cg1 : pc[0].cg2);
        const float g1 = e1[c] * (oldc ? pc[1].cg1 : pc[1].cg2);
        if (c < K) Raw<T>::st(col + (size_t)c * kBox, g0, g1);
      }
      // the label's own channel: recomputed in fp32 so that -dy is applied before rounding
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (y[j] >= 0 && pc[j].dy != 0.f) {
          const int kk = y[j];
          const float cgk = kk == 0 ? pc[j].cg0 : (kk < old_cl ? pc[j].cg1 : pc[j].cg2);
          const float ey = ex2_fast(fmaf(xy[j], kLog2e, j == 0 ? nm0 : nm1));
          col[(size_t)kk * kBox + j] = DT<T>::from_f(ey * cgk - pc[j].dy - (kk == 0 ? pc[j].d0 : 0.f));
        }
      }
      fence_proxy_async();
    }
    mbar_arrive(&bar_done[s]);

    // ---- issuing lane: write tile k-1 back, refill the stage of tile k-2 with tile k+2 (both
    //      conditions were met a whole tile ago, so nothing here blocks) ---------------------------------
    if (issuer) {
      if (k >= 1) {
        // every thread has written its gradients of tile k-1 (and finished reading tile k-2)
        mbar_wait(&bar_done[(k - 1) % S], (uint32_t)(((k - 1) / S) & 1));
        if (a.dlogits) {
          issue_store(sb, st, (k - 1) % S);
          advance(sb, st);
          // the store of tile k-2 (issued one tile ago) has finished reading its stage
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        }
      }
      if (k + 2 < my_tiles) {
        issue_load(pb, pt, (k + 2) % S);
        advance(pb, pt);
      }
    }
    __syncwarp();

    // ---- arg-max / mask stores -------------------------------------------------------------------------
    if (a.preds)
      *reinterpret_cast<longlong2*>(a.preds + (int64_t)b * HW + p0 + px0) = make_longlong2((long long)am0, (long long)am1);
    if (a.distill_mask)
      *reinterpret_cast<uchar2*>(a.distill_mask + (int64_t)b * HW + p0 + px0) = make_uchar2(dmask[0], dmask[1]);

    // ---- focal gradient: adjoint of the bilinear up-sample, reduced per warp ------------------------------
    if (a.gz) {
      const unsigned full = 0xffffffffu;
      if (ROWTILE) {
        // the warp's pixels share the row weights: reduce (g*(1-wx), g*wx) over runs of equal low-res column
        float c0 = gfoc[0] * (1.f - wx1[0]), c1 = gfoc[0] * wx1[0];
        const int key = cx0[0] * 2 + cdx[0];
        float d0 = 0.f, d1 = 0.f;
        int x2 = -1, dx2 = 0;
        {
          const float f0 = gfoc[1] * (1.f - wx1[1]), f1 = gfoc[1] * wx1[1];
          if (cx0[1] * 2 + cdx[1] == key) {
            c0 += f0;
            c1 += f1;
          } else {  // low-res column boundary inside the pair
            d0 = f0; d1 = f1; x2 = cx0[1]; dx2 = cdx[1];
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
        float* g0p = a.gz + (int64_t)b * a.h * a.w + ly_row.i0 * a.w;
        float* g1p = a.gz + (int64_t)b * a.h * a.w + ly_row.i1 * a.w;
        const float wy0 = 1.f - ly_row.w1, wy1 = ly_row.w1;
        if (((lane == 0) || (pk != key)) && cx0[0] >= 0) {
          if (c0 != 0.f) {
            atomicAdd(g0p + cx0[0], wy0 * c0);
            if (wy1 != 0.f) atomicAdd(g1p + cx0[0], wy1 * c0);
          }
          if (c1 != 0.f) {
            atomicAdd(g0p + cx0[0] + cdx[0], wy0 * c1);
            if (wy1 != 0.f) atomicAdd(g1p + cx0[0] + cdx[0], wy1 * c1);
          }
        }
        if (x2 >= 0) {
          if (d0 != 0.f) {
            atomicAdd(g0p + x2, wy0 * d0);
            if (wy1 != 0.f) atomicAdd(g1p + x2, wy1 * d0);
          }
          if (d1 != 0.f) {
            atomicAdd(g0p + x2 + dx2, wy0 * d1);
            if (wy1 != 0.f) atomicAdd(g1p + x2 + dx2, wy1 * d1);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
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

    if (a.mode == BACS_PIX_SCORE) {  // per-image sums: flush the accumulators per tile
#pragma unroll
      for (int i = 0; i < BACS_NACC; ++i) {
        const float r = warp_sum(acc[i]);
        if (lane == 0) red_scratch[wid][i] = r;
        acc[i] = 0.f;
      }
      fast_sync();
      if (tid < BACS_NACC) {
        float r = 0.f;
        for (int wv = 0; wv < 8; ++wv) r += red_scratch[wv][tid];
        p.partials[((int64_t)b * tpi + t_in) * BACS_NACC + tid] = (double)r;
      }
      fast_sync();
    }
  }
  if (issuer && my_tiles > 0) {  // the last tile's gradient rows
    const int kl = my_tiles - 1;
    mbar_wait(&bar_done[kl % S], (uint32_t)((kl / S) & 1));
    if (a.dlogits) issue_store(sb, st, kl % S);
    bulk_wait_all();
  }

  if (a.mode != BACS_PIX_SCORE) {
#pragma unroll
    for (int i = 0; i < BACS_NACC; ++i) {
      const float r = warp_sum(acc[i]);
      if (lane == 0) red_scratch[wid][i] = r;
    }
    fast_sync();
    if (tid < BACS_NACC) {
      double r = 0.0;
      for (int wv = 0; wv < 8; ++wv) r += (double)red_scratch[wv][tid];
      p.partials[(int64_t)blockIdx.x * BACS_NACC + tid] = r;
    }
  }
}

template <typename T, int KREG, bool ROWTILE>
static int launch_fast_one(const PixelParams& p, const PixelPlan& plan, cudaStream_t s) {
  return launch_pixel_kernel("bacs_pixel_loss", false, pixel_fast_kernel<T, KREG, ROWTILE>, dim3(plan.grid),
                             dim3(kFastThreads), plan.smem, s, p);
}

template <typename T>
static int launch_fast_dtype(const PixelParams& p, const PixelPlan& plan, cudaStream_t s) {
#define BACS_FAST_CASE(KR)                                             \
  case KR:                                                             \
    return plan.rowtile ? launch_fast_one<T, KR, true>(p, plan, s)     \
                        : launch_fast_one<T, KR, false>(p, plan, s);
  switch (plan.kreg) {
    BACS_FAST_CASE(4)
    BACS_FAST_CASE(8)
    BACS_FAST_CASE(12)
    BACS_FAST_CASE(16)
    BACS_FAST_CASE(20)
    BACS_FAST_CASE(21)
    BACS_FAST_CASE(24)
    default:
      set_error("bacs_pixel_loss: no fast kernel for KREG=%d", plan.kreg);
      return BACS_ERR_UNSUPPORTED;
  }
#undef BACS_FAST_CASE
}

}  // namespace bacs
